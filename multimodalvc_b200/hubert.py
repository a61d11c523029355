"""Host-side mirror of the reference's ``AVHubertModel`` for the encoder hot path (avhubert/hubert.py:334-779).

Same constructor shape (``AVHubertModel(cfg, task_cfg, dictionaries)`` / ``build_model(cfg, task)``), same
state-dict key names (so ``load_state_dict(state["model"], strict=False)`` from a reference checkpoint works:
src/model.py:223-224, avhubert/hubert_asr.py:303), same ``extract_finetune`` signature, tensor layouts,
padding-mask semantics and ``[B,T,D]`` output (avhubert/hubert.py:694-745).  The torch modules below are
*parameter containers only* — their ``forward`` is never called.  All arithmetic happens in
``libavh_b200.so`` (hand-written sm_100a kernels) through the C ABI in ``include/avh_b200.h``; there is no
PyTorch or CPU fallback, and calls fail loudly when the extension is missing or the tensors are not on a
B200-class device.
"""
import ctypes
import math
from dataclasses import dataclass, field
from typing import Optional

import numpy as np
import torch
import torch.nn as nn

from . import _lib, masking
from ._train import StepRegularization, backward_flat, refresh_weights_device

_DTYPES = {torch.float32: _lib.AVH_F32, torch.float16: _lib.AVH_F16, torch.bfloat16: _lib.AVH_BF16}
_U8 = _lib.AVH_U8        # raw uint8 video frames (normalised + centre-cropped on the device)


@dataclass
class AVHubertConfig:
    """The fields of the reference ``AVHubertConfig`` (avhubert/hubert.py:64-315) that shape this path, with the
    reference defaults.  Pretraining-only fields are accepted (kept as attributes) and ignored."""
    label_rate: int = 25
    encoder_layers: int = 12
    encoder_embed_dim: int = 768
    encoder_ffn_embed_dim: int = 3072
    encoder_attention_heads: int = 12
    activation_fn: str = "gelu"
    dropout: float = 0.1
    attention_dropout: float = 0.1
    activation_dropout: float = 0.0
    encoder_layerdrop: float = 0.0
    dropout_input: float = 0.0
    dropout_features: float = 0.0
    final_dim: int = 0
    untie_final_proj: bool = False
    layer_norm_first: bool = False
    feature_grad_mult: float = 1.0
    conv_pos: int = 128
    conv_pos_groups: int = 16
    resnet_relu_type: str = "prelu"
    resnet_weights: Optional[str] = None
    sub_encoder_layers: int = 0
    audio_feat_dim: int = -1
    modality_dropout: float = 0.0
    audio_dropout: float = 0.0
    modality_fuse: str = "concat"
    masking_type: str = "input"
    # span masking / masked-prediction head (pretraining-mode forward; avhubert/hubert.py:146-258 defaults)
    logit_temp: float = 0.1
    target_glu: bool = False
    mask_length_audio: int = 10
    mask_prob_audio: float = 0.65
    mask_length_image: int = 10
    mask_prob_image: float = 0.65
    mask_selection: str = "static"
    mask_other: float = 0
    no_mask_overlap: bool = False
    mask_min_space: int = 1
    mask_channel_length: int = 10
    mask_channel_prob: float = 0.0
    mask_channel_selection: str = "static"
    mask_channel_other: float = 0
    no_mask_channel_overlap: bool = False
    mask_channel_min_space: int = 1
    skip_masked: bool = False
    skip_nomask: bool = False
    sim_type: str = "cosine"
    selection_type: str = "same_other_seq"
    # --- B200 build options (not in the reference) ---
    compute_dtype: str = "auto"        # "auto": fp32 module -> fp32-faithful mode, half/bf16 module -> bf16 mode
    frontend_chunk_frames: int = 0     # 0 = library default
    capture_stages: bool = False       # keep intermediate stages readable (tests)
    trainable: bool = False            # also pack the backward's operands: extract_finetune in .train() with gradients
                                       # enabled differentiates the tail (fusion LayerNorm, post_extract_proj, encoder)
    ragged: str = "dense"              # "dense": compute on the padded [B,T] batch, every output position as the
                                       # reference's; "packed": bf16 mode, frames/tokens of ragged batches packed back to
                                       # back (no work on pad frames), output rows at pad positions are zeros

    @staticmethod
    def named(size, **kw):
        """Shipped shapes: Base (avhubert/conf/pretrain/base_vox_iter5.yaml:70-97) and Large
        (large_vox_iter5.yaml:70-101); `tiny` is a test-sized shape with the same structure."""
        shape = dict(base=(12, 768, 3072, 12), large=(24, 1024, 4096, 16), tiny=(2, 128, 256, 2))[size]
        cfg = AVHubertConfig(encoder_layers=shape[0], encoder_embed_dim=shape[1], encoder_ffn_embed_dim=shape[2],
                             encoder_attention_heads=shape[3], audio_feat_dim=104, layer_norm_first=True)
        for k, v in kw.items():
            setattr(cfg, k, v)
        return cfg


# ----------------------------------------------------------------------------- parameter containers
class _BasicBlockParams(nn.Module):      # avhubert/resnet.py:35-74
    def __init__(self, cin, cout, stride):
        super().__init__()
        self.conv1 = nn.Conv2d(cin, cout, 3, stride, 1, bias=False)
        self.bn1 = nn.BatchNorm2d(cout)
        self.relu1 = nn.PReLU(num_parameters=cout)
        self.relu2 = nn.PReLU(num_parameters=cout)
        self.conv2 = nn.Conv2d(cout, cout, 3, 1, 1, bias=False)
        self.bn2 = nn.BatchNorm2d(cout)
        self.downsample = None
        if stride != 1 or cin != cout:   # downsample_basic_block, resnet.py:20-24
            self.downsample = nn.Sequential(nn.Conv2d(cin, cout, 1, stride, bias=False), nn.BatchNorm2d(cout))


class _TrunkParams(nn.Module):           # avhubert/resnet.py:77-129, layers [2,2,2,2]
    def __init__(self):
        super().__init__()
        cin = 64
        for i, w in enumerate([64, 128, 256, 512]):
            stride = 1 if i == 0 else 2
            setattr(self, f"layer{i + 1}", nn.Sequential(_BasicBlockParams(cin, w, stride), _BasicBlockParams(w, w, 1)))
            cin = w
        for m in self.modules():         # resnet.py:92-98
            if isinstance(m, nn.Conv2d):
                n = m.kernel_size[0] * m.kernel_size[1] * m.out_channels
                m.weight.data.normal_(0, math.sqrt(2.0 / n))


class _ResEncoderParams(nn.Module):      # avhubert/resnet.py:131-142
    backend_out = 512

    def __init__(self):
        super().__init__()
        self.frontend3D = nn.Sequential(
            nn.Conv3d(1, 64, (5, 7, 7), (1, 2, 2), (2, 3, 3), bias=False), nn.BatchNorm3d(64), nn.PReLU(num_parameters=64),
            nn.MaxPool3d((1, 3, 3), (1, 2, 2), (0, 1, 1)))
        self.trunk = _TrunkParams()


class _SubModelParams(nn.Module):        # avhubert/hubert.py:317-332 (sub_encoder_layers == 0)
    def __init__(self, resnet, input_dim, dim):
        super().__init__()
        self.resnet = resnet
        self.proj = nn.Linear(input_dim, dim)
        self.encoder = None


class _PosConvParams(nn.Module):         # weight_norm(Conv1d, dim=2): wav2vec2.py:822-834
    def __init__(self, dim, k, groups):
        super().__init__()
        std = math.sqrt(4.0 / (k * dim))
        v = torch.randn(dim, dim // groups, k) * std
        self.weight_g = nn.Parameter(v.norm(dim=(0, 1), keepdim=True).clone())
        self.weight_v = nn.Parameter(v)
        self.bias = nn.Parameter(torch.zeros(dim))


class _SelfAttnParams(nn.Module):        # fairseq/fairseq/modules/multihead_attention.py:64-77
    def __init__(self, dim):
        super().__init__()
        self.k_proj = nn.Linear(dim, dim)
        self.v_proj = nn.Linear(dim, dim)
        self.q_proj = nn.Linear(dim, dim)
        self.out_proj = nn.Linear(dim, dim)


class _LayerParams(nn.Module):           # wav2vec2.py:907-958
    def __init__(self, dim, ffn):
        super().__init__()
        self.self_attn = _SelfAttnParams(dim)
        self.self_attn_layer_norm = nn.LayerNorm(dim)
        self.fc1 = nn.Linear(dim, ffn)
        self.fc2 = nn.Linear(ffn, dim)
        self.final_layer_norm = nn.LayerNorm(dim)


class _EncoderParams(nn.Module):         # wav2vec2.py:816-857
    def __init__(self, cfg):
        super().__init__()
        D = cfg.encoder_embed_dim
        self.embedding_dim = D
        self.layer_norm_first = cfg.layer_norm_first
        self.pos_conv = nn.Sequential(_PosConvParams(D, cfg.conv_pos, cfg.conv_pos_groups))
        self.layers = nn.ModuleList([_LayerParams(D, cfg.encoder_ffn_embed_dim) for _ in range(cfg.encoder_layers)])
        self.layer_norm = nn.LayerNorm(D)
        for m in self.modules():         # init_bert_params
            if isinstance(m, nn.Linear):
                m.weight.data.normal_(0.0, 0.02)
                m.bias.data.zero_()


class _TailTrainFn(torch.autograd.Function):
    """y = encoder(post_extract_proj(layer_norm(fused))) with the library's forward (activations saved in the plan) and
    backward; the parameters are arguments only so that autograd routes their gradients."""

    @staticmethod
    def forward(ctx, model, reg, fused, pm_u8, *params):
        handle = model._ensure_handle()
        dev = fused.device
        B, T, _ = fused.shape
        out_dtype = model.encoder.layer_norm.weight.dtype
        if out_dtype not in _DTYPES:
            out_dtype = torch.float32
        out = torch.empty(B, T, model.encoder_embed_dim, device=dev, dtype=out_dtype)
        fused = fused.contiguous()
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            reg.set_on(handle)
            _lib.check(_lib.load().avh_tail_train_forward(
                handle, ctypes.c_void_p(fused.data_ptr()), _DTYPES[fused.dtype],
                ctypes.c_void_p(pm_u8.data_ptr()) if pm_u8 is not None else None, B, T,
                ctypes.c_void_p(out.data_ptr()), _DTYPES[out_dtype], ctypes.c_void_p(stream)))
        ctx.handle, ctx.stream, ctx.model, ctx.params, ctx.reg = handle, stream, model, params, reg
        ctx.shapes = [tuple(p.shape) for p in params]
        ctx.dtypes = [p.dtype for p in params]
        return out

    @staticmethod
    def backward(ctx, dout):
        dev = dout.device
        dout = dout.contiguous()
        if dout.dtype not in _DTYPES:
            dout = dout.float()
        lib = _lib.load()
        n = ctypes.c_int64()
        _lib.check(lib.avh_tail_grad_count(ctx.handle, ctypes.byref(n)))
        flat = backward_flat(ctx.handle, dout, None, n.value, ctx.dtypes, ctx.stream, ctx.model)
        grads, off = [], 0
        for shape, dt in zip(ctx.shapes, ctx.dtypes):
            k = 1
            for d in shape:
                k *= d
            grads.append(flat.of(dt)[off:off + k].view(shape))
            off += k
        assert off == n.value
        if flat.reduced:
            ctx.model._grad_sync.mark_reduced(ctx.params)
        return (None, None, None, None, *ctx.reg.layer_grads(grads, flat.reduced))


class _FullTrainFn(torch.autograd.Function):
    """The whole fine-tuning step (feature_grad_mult > 0): lip ResNet + projections + fusion + encoder with the library's
    forward (activations saved in the plan) and backward; `spec` = [(buffer shape, to_param)] describes how the flat
    gradient buffer maps onto the parameters that follow."""

    @staticmethod
    def forward(ctx, model, reg, video, audio, pm_u8, fgm, spec, *params):
        handle = model._ensure_handle()
        ref = video if video is not None else audio
        dev = ref.device
        B, T = (video.size(0), video.size(2)) if video is not None else (audio.size(0), audio.size(2))
        out_dtype = model.encoder.layer_norm.weight.dtype
        if out_dtype not in _DTYPES:
            out_dtype = torch.float32
        out = torch.empty(B, T, model.encoder_embed_dim, device=dev, dtype=out_dtype)
        strides = (ctypes.c_int64 * 3)(*audio.stride()) if audio is not None else None
        vp = ctypes.c_void_p
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            reg.set_on(handle)
            _lib.check(_lib.load().avh_full_train_forward(
                handle, vp(video.data_ptr()) if video is not None else None, _DTYPES[video.dtype] if video is not None else 0,
                vp(audio.data_ptr()) if audio is not None else None, _DTYPES[audio.dtype] if audio is not None else 0, strides,
                vp(pm_u8.data_ptr()) if pm_u8 is not None else None, B, T, float(fgm), 0.1, vp(out.data_ptr()),
                _DTYPES[out_dtype], vp(stream)))
        ctx.handle, ctx.stream, ctx.spec, ctx.reg = handle, stream, spec, reg
        ctx.model, ctx.params = model, params
        ctx.flags = (int(video is not None), int(audio is not None))
        ctx.keep = (video, audio)                      # the backward re-reads the frames (stem patches are recomputed)
        ctx.dtypes = [p.dtype for p in params]
        return out

    @staticmethod
    def backward(ctx, dout):
        dev = dout.device
        dout = dout.contiguous()
        if dout.dtype not in _DTYPES:
            dout = dout.float()
        lib = _lib.load()
        n = ctypes.c_int64()
        _lib.check(lib.avh_full_grad_count(ctx.handle, ctx.flags[0], ctx.flags[1], ctypes.byref(n)))
        flat = backward_flat(ctx.handle, dout, None, n.value, ctx.dtypes, ctx.stream, ctx.model)
        grads, off = [], 0
        for (shape, to_param), dt in zip(ctx.spec, ctx.dtypes):
            k = 1
            for d in shape:
                k *= d
            grads.append(to_param(flat.of(dt)[off:off + k].view(shape)))
            off += k
        assert off == n.value, (off, n.value)
        if flat.reduced:
            ctx.model._grad_sync.mark_reduced(ctx.params)
        return (None, None, None, None, None, None, None, *ctx.reg.layer_grads(grads, flat.reduced))


class AVHubertModel(nn.Module):
    """Drop-in for the reference ``AVHubertModel`` on the ``extract_finetune`` path."""

    def __init__(self, cfg: AVHubertConfig, task_cfg=None, dictionaries=(None,), **kwargs):
        super().__init__()
        if cfg.activation_fn != "gelu":
            raise NotImplementedError("only activation_fn='gelu' (every shipped AV-HuBERT config) is implemented")
        if cfg.sub_encoder_layers != 0:
            raise NotImplementedError("sub_encoder_layers > 0 is not used by any shipped config")
        if cfg.resnet_relu_type != "prelu":
            raise NotImplementedError("only resnet_relu_type='prelu' is implemented")
        if cfg.modality_fuse not in ("concat", "add"):
            raise ValueError(f"unknown modality_fuse {cfg.modality_fuse}")
        if cfg.audio_feat_dim <= 0:
            raise ValueError("audio_feat_dim must be set (104 for 4x26 stacked log-fbank)")
        self.cfg = cfg
        D = cfg.encoder_embed_dim
        self.encoder_embed_dim = D
        self.modality_fuse = cfg.modality_fuse
        self.embed = 2 * D if cfg.modality_fuse == "concat" else D
        self.feature_extractor_audio = _SubModelParams(None, cfg.audio_feat_dim, D)
        self.feature_extractor_video = _SubModelParams(_ResEncoderParams(), _ResEncoderParams.backend_out, D)
        self.post_extract_proj = nn.Linear(self.embed, D) if self.embed != D else None
        self.mask_emb = nn.Parameter(
            torch.FloatTensor(cfg.audio_feat_dim if cfg.masking_type == "input" else D).uniform_())
        self.encoder = _EncoderParams(cfg)
        self.layer_norm = nn.LayerNorm(self.embed)
        final_dim = cfg.final_dim if cfg.final_dim > 0 else D
        if cfg.target_glu:
            raise NotImplementedError("target_glu is false in every shipped config (and unused by the reference forward)")
        dictionaries = list(dictionaries) if dictionaries is not None else [None]
        # pretraining head (hubert.py:409-426); dropped by remove_pretraining_modules
        self.untie_final_proj = bool(cfg.untie_final_proj)
        self.final_proj = nn.Linear(D, final_dim * (len(dictionaries) if self.untie_final_proj else 1))
        self.num_classes = None
        if not any(d is None for d in dictionaries):
            self.num_classes = [len(d) for d in dictionaries]
            self.label_embs_concat = nn.Parameter(torch.FloatTensor(sum(self.num_classes), final_dim).uniform_())
        sample_rate = getattr(task_cfg, "sample_rate", cfg.label_rate) if task_cfg is not None else cfg.label_rate
        self.feat2tar_ratio = cfg.label_rate / sample_rate          # hubert.py:346-347 (feature_ds_rate = 1)
        self._handle = None
        self._handle_key = None
        self._dirty = True
        self._video_geo = None
        self._eval_stale = False
        self._host_keepalive = {}
        self._param_versions = None
        # normalisation of raw uint8 video (task config image_mean / image_std, hubert_pretraining.py:144-149)
        self.image_mean, self.image_std = 0.421, 0.165
        self.register_load_state_dict_post_hook(lambda module, incompatible: module._mark_dirty())

    # ------------------------------------------------------------------ reference API surface
    @classmethod
    def build_model(cls, cfg: AVHubertConfig, task=None):
        """avhubert/hubert.py:434-440"""
        return cls(cfg, getattr(task, "cfg", None), getattr(task, "dictionaries", (None,)))

    def upgrade_state_dict_named(self, state_dict, name):
        return state_dict

    def remove_pretraining_modules(self):
        """avhubert/hubert.py:757-759"""
        self.target_glu = None
        self.final_proj = None

    @staticmethod
    def forward_padding_mask(features_len: int, padding_mask: torch.Tensor) -> torch.Tensor:
        """avhubert/hubert.py:564-574 (identity when the mask already has one entry per frame)."""
        extra = padding_mask.size(1) % features_len
        if extra > 0:
            padding_mask = padding_mask[:, :-extra]
        padding_mask = padding_mask.view(padding_mask.size(0), features_len, -1)
        return padding_mask.all(-1)

    # ------------------------------------------------------------------ weights -> device library
    def _mark_dirty(self):
        self._dirty = True

    def _apply(self, fn, *args, **kwargs):       # .cuda() / .half() / .to(): packed copies become stale
        out = super()._apply(fn, *args, **kwargs)
        self._dirty = True
        return out

    def refresh_weights(self):
        """Call after modifying parameters in place (optimizer step, manual edits)."""
        self._dirty = True

    def _sync_trained_weights(self):
        """Training steps: when an optimizer step changed the parameters since the last forward, refresh the packed
        copies the training plans read — on the device, in place (a few ms; the full re-pack through the host takes
        seconds for Large).  The eval-only packed forms are left stale: the next eval forward re-packs everything."""
        versions = [p._version for p in self.parameters()]
        if self._param_versions == versions:
            return
        if self._handle is not None and not self._dirty and self._param_versions is not None:
            refresh_weights_device(self._handle, self)
            self._eval_stale = True
        else:
            self._dirty = True
        self._param_versions = versions

    def _destroy_handle(self):
        if self._handle is not None:
            _lib.load().avh_destroy(self._handle)
            self._handle = None
            self._handle_key = None
            self._video_geo = None

    def __del__(self):
        try:
            self._destroy_handle()
        except Exception:
            pass

    def _compute_mode(self, dtype):
        cd = self.cfg.compute_dtype
        if cd == "auto":
            return _lib.AVH_COMPUTE_FP32 if dtype == torch.float32 else _lib.AVH_COMPUTE_BF16
        if cd in ("bf16", "bfloat16"):
            return _lib.AVH_COMPUTE_BF16
        if cd in ("fp32", "float32"):
            return _lib.AVH_COMPUTE_FP32
        raise ValueError(f"compute_dtype must be auto|bf16|fp32, got {cd}")

    def _ensure_handle(self):
        p = self.encoder.layer_norm.weight
        if p.device.type != "cuda":
            raise RuntimeError("multimodalvc_b200.AVHubertModel computes on a B200 only: move the module to a CUDA "
                               "device (there is no CPU path)")
        key = (p.device.index if p.device.index is not None else torch.cuda.current_device(),
               self._compute_mode(p.dtype))
        if not self.training and getattr(self, "_eval_stale", False):
            # training moved the BatchNorm running statistics / a device-side refresh skipped the eval-only packed forms
            self._dirty, self._eval_stale = True, False
        if self._handle is not None and key == self._handle_key and not self._dirty:
            return self._handle
        lib = _lib.load()
        if self._handle is None or key != self._handle_key:
            self._destroy_handle()
            c = self.cfg
            cc = _lib.AvhConfig(
                encoder_layers=c.encoder_layers, encoder_embed_dim=c.encoder_embed_dim,
                encoder_ffn_embed_dim=c.encoder_ffn_embed_dim, encoder_attention_heads=c.encoder_attention_heads,
                audio_feat_dim=c.audio_feat_dim,
                modality_fuse=_lib.AVH_FUSE_CONCAT if c.modality_fuse == "concat" else _lib.AVH_FUSE_ADD,
                layer_norm_first=int(bool(c.layer_norm_first)), conv_pos=c.conv_pos, conv_pos_groups=c.conv_pos_groups,
                compute_mode=key[1], frontend_chunk_frames=int(c.frontend_chunk_frames),
                capture_stages=int(bool(c.capture_stages)))
            cc.reserved[3] = 1 if c.trainable else 0
            hp = ctypes.c_void_p()
            _lib.check(lib.avh_create(ctypes.byref(cc), key[0], ctypes.byref(hp)))
            self._handle, self._handle_key = hp, key
        with torch.no_grad():
            for name, t in self.state_dict().items():
                if (name in ("mask_emb", "label_embs_concat") or name.startswith("final_proj.")
                        or name.endswith("num_batches_tracked")):
                    continue
                if not t.is_floating_point():
                    continue
                t = t.detach().contiguous()
                if t.dtype not in _DTYPES:
                    t = t.float()
                shape = (ctypes.c_int64 * max(t.dim(), 1))(*t.shape)
                _lib.check(lib.avh_load_tensor(self._handle, name.encode(), ctypes.c_void_p(t.data_ptr()),
                                               _DTYPES[t.dtype], shape, t.dim()))
            torch.cuda.synchronize(p.device)
        _lib.check(lib.avh_finalize_weights(self._handle))
        # every refresh re-loads the whole state dict, so the library's fp32 host copies (1.3 GB for Large) can go
        _lib.check(lib.avh_drop_host_weights(self._handle))
        self._dirty = False
        return self._handle

    # ------------------------------------------------------------------ the hot path
    def _check_mode(self, mask, allow_train=False):
        if mask:
            raise NotImplementedError("span masking is applied by extract_finetune / extract_features / forward on "
                                      "device tensors only")
        if self.training and not allow_train:
            raise RuntimeError("this entry point runs the eval-mode forward only; call .eval() (extract_finetune on "
                               "device tensors supports the training-mode forward)")

    def _bn_modules(self):
        """BatchNorm modules in the order avh_read_bn_stats writes their running statistics."""
        res = self.feature_extractor_video.resnet
        out = [res.frontend3D[1]]
        for i in range(1, 5):
            for blk in getattr(res.trunk, f"layer{i}"):
                out += [blk.bn1, blk.bn2]
                if blk.downsample is not None:
                    out.append(blk.downsample[1])
        return out

    def _train_args(self, output_layer, regularise=True):
        """Per-call arguments of the training-mode forward: dropout probabilities of the config, a seed from torch's
        CPU generator, and the LayerDrop coins — drawn with np.random.random() in layer order up to the exit layer,
        exactly as the reference does (wav2vec2.py:886-888), so the same numpy seed drops the same layers.
        regularise=False: no dropout, no layer dropped, nothing drawn (a pass that only reads an early stage)."""
        import numpy as np
        c = self.cfg
        if not regularise:
            skip_arr = (ctypes.c_uint8 * c.encoder_layers)()
            ta = _lib.AvhTrainArgs(dropout_input=0.0, dropout=0.0, activation_dropout=0.0, attention_dropout=0.0,
                                   bn_momentum=0.1, seed=0, layer_skip=ctypes.cast(skip_arr, ctypes.c_void_p))
            return ta, skip_arr, [0] * c.encoder_layers
        if c.attention_dropout > 0:
            raise NotImplementedError("attention_dropout > 0 in training mode is not implemented (0.0 in every "
                                      "shipped fine-tune config, avhubert/conf/finetune/*.yaml)")
        n = c.encoder_layers if output_layer is None else min(int(output_layer), c.encoder_layers)
        skip = [0] * c.encoder_layers
        for i in range(n):
            skip[i] = 0 if np.random.random() > c.encoder_layerdrop else 1
        skip_arr = (ctypes.c_uint8 * c.encoder_layers)(*skip)
        seed = int(torch.randint(0, 2 ** 62, (1,)).item())
        ta = _lib.AvhTrainArgs(dropout_input=float(c.dropout_input), dropout=float(c.dropout),
                               activation_dropout=float(c.activation_dropout), attention_dropout=0.0, bn_momentum=0.1,
                               seed=seed, layer_skip=ctypes.cast(skip_arr, ctypes.c_void_p))
        return ta, skip_arr, skip

    def _check_inputs(self, handle, src_video, src_audio, padding_mask, device):
        """Validation shared by the device and the host entry points.  Returns (video, video_dt, audio, pm_u8, pm, B, T)
        with video/audio contiguous-or-strided tensors on `device` ('cpu' for the host path) in a dtype the library
        reads, and pm the [B,T] bool mask (forward_padding_mask applied) or None."""
        if src_audio is None and src_video is None:
            raise ValueError("both modalities are None")
        for t in (src_video, src_audio):
            if t is not None and t.device != device:
                raise RuntimeError(f"inputs are on {t.device} but this call expects {device}")
        ref = src_video if src_video is not None else src_audio
        B, T = ref.size(0), -1
        video_dt = 0
        if src_video is not None:
            if src_video.dim() != 5 or src_video.size(1) != 1:
                raise ValueError(f"video must be [B,1,T,88,88] (or raw uint8 [B,1,T,H,W]), got {tuple(src_video.shape)}")
            T = src_video.size(2)
            if src_video.dtype == torch.uint8:
                # raw gray frames [B,1,T,H,W]: normalised and centre-cropped on the device (video.py)
                if min(src_video.shape[3:]) < 88:
                    raise ValueError(f"uint8 video must be [B,1,T,H>=88,W>=88], got {tuple(src_video.shape)}")
                self._set_video_geometry(handle, int(src_video.size(3)), int(src_video.size(4)))
                video_dt = _U8
            elif tuple(src_video.shape[3:]) != (88, 88):
                raise ValueError(f"video must be [B,1,T,88,88], got {tuple(src_video.shape)}")
            src_video = src_video.contiguous()
            if video_dt != _U8:
                if src_video.dtype not in _DTYPES:
                    src_video = src_video.float()
                video_dt = _DTYPES[src_video.dtype]
        if src_audio is not None:
            if src_audio.dim() != 3 or src_audio.size(1) != self.cfg.audio_feat_dim:
                raise ValueError(f"audio must be [B,{self.cfg.audio_feat_dim},T], got {tuple(src_audio.shape)}")
            if src_video is not None and (src_audio.size(2) != T or src_audio.size(0) != B):
                raise ValueError("audio and video disagree on batch/time")
            T = src_audio.size(2)
            if src_audio.dtype not in _DTYPES:
                src_audio = src_audio.float()
        if B < 1 or T < 1:
            raise ValueError("empty batch")
        pm_u8 = None
        if padding_mask is not None:
            if padding_mask.dim() != 2 or padding_mask.size(0) != B:
                raise ValueError(f"padding_mask must be [B,T'], got {tuple(padding_mask.shape)}")
            if padding_mask.size(1) != T:
                padding_mask = self.forward_padding_mask(T, padding_mask)
            pm_u8 = padding_mask.to(device=device, dtype=torch.bool).contiguous().view(torch.uint8)
        return src_video, video_dt, src_audio, pm_u8, padding_mask, B, T

    @staticmethod
    def lengths_from_padding_mask(padding_mask):
        """Valid frames per clip of a collater-style mask (True = padded, padding is a suffix: hubert_dataset.py:433-447)
        as a python list, or None when the mask is not of that form (padding inside a clip, an empty clip).  A CUDA mask
        costs one device->host copy; pass `lengths=` to extract_finetune to avoid it."""
        pm = padding_mask.detach().to("cpu", torch.bool)
        if pm.size(1) > 1 and not bool((pm[:, 1:] >= pm[:, :-1]).all()):
            return None
        lengths = (~pm).sum(1).tolist()
        return lengths if min(lengths) >= 1 else None

    def tail_parameters(self):
        """Parameters of the trainable tail in the order avh_encoder_backward writes their gradients."""
        out = []
        for layer in self.encoder.layers:
            a = layer.self_attn
            out += [a.q_proj.weight, a.k_proj.weight, a.v_proj.weight, a.q_proj.bias, a.k_proj.bias, a.v_proj.bias,
                    a.out_proj.weight, a.out_proj.bias, layer.self_attn_layer_norm.weight, layer.self_attn_layer_norm.bias,
                    layer.fc1.weight, layer.fc1.bias, layer.fc2.weight, layer.fc2.bias,
                    layer.final_layer_norm.weight, layer.final_layer_norm.bias]
        out += [self.encoder.layer_norm.weight, self.encoder.layer_norm.bias]
        pc = self.encoder.pos_conv[0]
        out += [pc.bias, pc.weight_g, pc.weight_v]
        if self.post_extract_proj is not None:
            out += [self.post_extract_proj.weight, self.post_extract_proj.bias]
        out += [self.layer_norm.weight, self.layer_norm.bias]
        return out

    def full_parameters(self, has_video, has_audio):
        """(parameters, spec) of the whole training step in the order avh_encoder_backward writes their gradients; spec =
        (shape of the gradient inside the flat buffer, map onto the parameter's own layout)."""
        same = lambda g: g
        params = self.tail_parameters()
        spec = [(tuple(p.shape), same) for p in params]
        D = self.encoder_embed_dim
        if has_audio:
            lin = self.feature_extractor_audio.proj
            Fa = lin.in_features
            Fp = (Fa + 63) // 64 * 64
            params += [lin.weight, lin.bias]
            spec += [((D, Fp), lambda g, Fa=Fa: g[:, :Fa]), ((D,), same)]
        if has_video:
            fe = self.feature_extractor_video
            params += [fe.proj.weight, fe.proj.bias]
            spec += [((D, 512), same), ((D,), same)]
            st = fe.resnet.frontend3D
            params += [st[0].weight, st[1].weight, st[1].bias, st[2].weight]
            spec += [((64, 5, 8, 8), lambda g: g[:, :, :7, :7].reshape(64, 1, 5, 7, 7)), ((64,), same), ((64,), same), ((64,), same)]
            cin = 64
            for i in range(1, 5):
                C = 64 << (i - 1)
                for blk in getattr(fe.resnet.trunk, f"layer{i}"):
                    params += [blk.conv1.weight, blk.bn1.weight, blk.bn1.bias, blk.relu1.weight,
                               blk.conv2.weight, blk.bn2.weight, blk.bn2.bias, blk.relu2.weight]
                    spec += [((C, 3, 3, cin), lambda g: g.permute(0, 3, 1, 2)), ((C,), same), ((C,), same), ((C,), same),
                             ((C, 3, 3, C), lambda g: g.permute(0, 3, 1, 2)), ((C,), same), ((C,), same), ((C,), same)]
                    if blk.downsample is not None:
                        params += [blk.downsample[0].weight, blk.downsample[1].weight, blk.downsample[1].bias]
                        spec += [((C, cin), lambda g, C=C, cin=cin: g.reshape(C, cin, 1, 1)), ((C,), same), ((C,), same)]
                    cin = C
        return params, spec

    def _step_regularization(self):
        c = self.cfg
        return StepRegularization(c.encoder_layers, dropout_input=c.dropout_input, dropout=c.dropout,
                                  activation_dropout=c.activation_dropout, attention_dropout=c.attention_dropout,
                                  layerdrop=c.encoder_layerdrop)

    def _extract_finetune_full(self, source, padding_mask, mask):
        """The whole model differentiable (feature_grad_mult > 0, hubert.py:538-547 with GradMultiply): SURVEY row A18 /
        BASELINE config 5 as stated."""
        c = self.cfg
        if mask and c.masking_type == "input":
            with torch.no_grad():
                v, _ = self.apply_input_mask(source["video"], padding_mask, None)
                a, _ = self.apply_input_mask(source["audio"], padding_mask, None)
            source = {"audio": a, "video": v}
        self._sync_trained_weights()
        handle = self._ensure_handle()
        self._param_versions = [p._version for p in self.parameters()]
        dev = self.encoder.layer_norm.weight.device
        video, video_dt, audio, pm_u8, pm, B, T = self._check_inputs(handle, source["video"], source["audio"], padding_mask, dev)
        if video is not None and video_dt == _U8:
            raise NotImplementedError("the training step takes normalised float video")
        params, spec = self.full_parameters(video is not None, audio is not None)
        reg = self._step_regularization()
        y = _FullTrainFn.apply(self, reg, video, audio, pm_u8, float(c.feature_grad_mult), spec, *params)
        self._last_train_args = (reg.seed, list(reg.skip))      # what the step used: tests rebuild its masks from it
        if video is not None:
            self._read_back_bn_stats(handle, dev)
        return y, pm

    @torch.no_grad()
    def _read_back_bn_stats(self, handle, dev):
        """Running statistics of the training-mode BatchNorms, updated on the device by the last forward, back into the
        module's buffers (the next eval forward folds them again)."""
        lib = _lib.load()
        n = ctypes.c_int64()
        _lib.check(lib.avh_bn_stats_count(handle, ctypes.byref(n)))
        flat = torch.empty(n.value, device=dev, dtype=torch.float32)
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            _lib.check(lib.avh_read_bn_stats(handle, ctypes.c_void_p(flat.data_ptr()), n.value, ctypes.c_void_p(stream)))
        off = 0
        for bn in self._bn_modules():
            C = bn.num_features
            bn.running_mean.copy_(flat[off:off + C])
            bn.running_var.copy_(flat[off + C:off + 2 * C])
            bn.num_batches_tracked += 1
            off += 2 * C
        self._eval_stale = True

    def _extract_finetune_trainable(self, source, padding_mask, mask, output_layer):
        """Fine-tuning step with frozen feature extractors (feature_grad_mult <= 0: the reference runs them under
        no_grad, hubert.py:538-547).  Extractors + fusion run as in the training-mode forward (batch-statistics
        BatchNorm), the fused features feed the differentiable tail: layer_norm -> post_extract_proj -> encoder."""
        c = self.cfg
        if output_layer is not None:
            raise NotImplementedError("the training step runs the whole encoder (output_layer=None)")
        if c.attention_dropout > 0:
            raise NotImplementedError("attention_dropout > 0 in training mode is not implemented (0.0 in every "
                                      "shipped fine-tune config, avhubert/conf/finetune/*.yaml)")
        if c.feature_grad_mult > 0:
            return self._extract_finetune_full(source, padding_mask, mask)
        self._sync_trained_weights()                             # an optimizer step changed the weights: refresh
        with torch.no_grad():
            # only the "fused" stage is read: no regularisation and no draws, so the step draws its coins once
            y1, pm = self._extract_finetune_nograd(source, padding_mask, mask=mask, output_layer=1, _regularise=False)
            B, T, _ = y1.shape
            fused = self.read_stage("fused", B * T * self.embed).view(B, T, self.embed)
        self._param_versions = [p._version for p in self.parameters()]
        dev = fused.device
        pm_u8 = pm.to(device=dev, dtype=torch.bool).contiguous().view(torch.uint8) if pm is not None else None
        reg = self._step_regularization()
        y = _TailTrainFn.apply(self, reg, fused, pm_u8, *self.tail_parameters())
        self._last_train_args = (reg.seed, list(reg.skip))      # what the step used: tests rebuild its masks from it
        return y, pm

    def extract_finetune(self, source, padding_mask=None, mask=False, ret_conv=False, output_layer=None, lengths=None):
        """avhubert/hubert.py:694-745 (see _extract_finetune_nograd).  In .train() with gradients enabled and
        cfg.trainable, the call is differentiable w.r.t. the tail's parameters (fusion LayerNorm, post_extract_proj,
        encoder): SURVEY row A18 with the feature extractors frozen."""
        if self.training and torch.is_grad_enabled() and self.cfg.trainable:
            return self._extract_finetune_trainable(source, padding_mask, mask, output_layer)
        return self._extract_finetune_nograd(source, padding_mask, mask=mask, ret_conv=ret_conv, output_layer=output_layer,
                                             lengths=lengths)

    @torch.no_grad()
    def _extract_finetune_nograd(self, source, padding_mask=None, mask=False, ret_conv=False, output_layer=None, lengths=None,
                                 _regularise=True):
        """avhubert/hubert.py:694-745.  source = {'audio': [B,F,T] | None, 'video': [B,1,T,88,88] | None};
        padding_mask bool [B,T] (True = padded).  Returns (x [B,T,D], padding_mask).  With cfg.ragged == "packed" (bf16
        mode) ragged batches run packed; `lengths` (valid frames per clip) may be given to skip reading the mask back."""
        if mask and self.cfg.masking_type == "input":
            # hubert.py:696-699: video first, then audio (the order fixes the RNG stream); the union is not used here
            src_video, _ = self.apply_input_mask(source["video"], padding_mask, None)
            src_audio, _ = self.apply_input_mask(source["audio"], padding_mask, None)
            source = {"audio": src_audio, "video": src_video}
        self._check_mode(False, allow_train=True)
        if not self.training and getattr(self, "_eval_stale", False):
            # training-mode forwards moved the BatchNorm running statistics: fold the current ones for eval
            self._dirty, self._eval_stale = True, False
        handle = self._ensure_handle()
        dev = self.encoder.layer_norm.weight.device
        src_video, video_dt, src_audio, pm_u8, padding_mask, B, T = self._check_inputs(
            handle, source["video"], source["audio"], padding_mask, dev)
        out_dtype = self.encoder.layer_norm.weight.dtype
        if out_dtype not in _DTYPES:
            out_dtype = torch.float32
        out = torch.empty(B, T, self.encoder_embed_dim, device=dev, dtype=out_dtype)
        strides = None
        if src_audio is not None:
            strides = (ctypes.c_int64 * 3)(*src_audio.stride())
        ol = 0 if output_layer is None else int(output_layer)
        if self.training:
            # frozen-encoder-in-train-mode forward (src/model.py:96-100,280): batch-statistics BatchNorm, dropout, LayerDrop
            if video_dt == _U8:
                raise NotImplementedError("the training-mode forward takes normalised float video")
            ta, skip_arr, _ = self._train_args(output_layer, regularise=_regularise)
            lib = _lib.load()
            with torch.cuda.device(dev):
                stream = torch.cuda.current_stream(dev).cuda_stream
                _lib.check(lib.avh_forward_train(
                    handle,
                    ctypes.c_void_p(src_video.data_ptr()) if src_video is not None else None, video_dt,
                    ctypes.c_void_p(src_audio.data_ptr()) if src_audio is not None else None,
                    _DTYPES[src_audio.dtype] if src_audio is not None else 0, strides,
                    ctypes.c_void_p(pm_u8.data_ptr()) if pm_u8 is not None else None,
                    B, T, ol, ctypes.byref(ta), ctypes.c_void_p(out.data_ptr()), _DTYPES[out_dtype], ctypes.c_void_p(stream)))
            if src_video is not None:
                self._read_back_bn_stats(handle, dev)
            return out, padding_mask
        if self.cfg.ragged not in ("dense", "packed"):
            raise ValueError(f"cfg.ragged must be 'dense' or 'packed', got {self.cfg.ragged}")
        if (self.cfg.ragged == "packed" and padding_mask is not None and self._handle_key[1] == _lib.AVH_COMPUTE_BF16):
            if lengths is None:
                lengths = self.lengths_from_padding_mask(padding_mask)
            elif len(lengths) != B or min(lengths) < 1 or max(lengths) > T:
                raise ValueError("lengths must hold one value in [1, T] per clip")
            if lengths is not None:
                with torch.cuda.device(dev):
                    stream = torch.cuda.current_stream(dev).cuda_stream
                    _lib.check(_lib.load().avh_forward_ragged(
                        handle,
                        ctypes.c_void_p(src_video.data_ptr()) if src_video is not None else None,
                        video_dt,
                        ctypes.c_void_p(src_audio.data_ptr()) if src_audio is not None else None,
                        _DTYPES[src_audio.dtype] if src_audio is not None else 0,
                        strides, (ctypes.c_int32 * B)(*[int(n) for n in lengths]),
                        B, T, ol, ctypes.c_void_p(out.data_ptr()), _DTYPES[out_dtype], ctypes.c_void_p(stream)))
                return out, padding_mask
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            _lib.check(_lib.load().avh_forward(
                handle,
                ctypes.c_void_p(src_video.data_ptr()) if src_video is not None else None,
                video_dt,
                ctypes.c_void_p(src_audio.data_ptr()) if src_audio is not None else None,
                _DTYPES[src_audio.dtype] if src_audio is not None else 0,
                strides,
                ctypes.c_void_p(pm_u8.data_ptr()) if pm_u8 is not None else None,
                B, T, ol, ctypes.c_void_p(out.data_ptr()), _DTYPES[out_dtype], ctypes.c_void_p(stream)))
        return out, padding_mask

    def _set_video_geometry(self, handle, H, W):
        geo = (H, W, float(self.image_mean), float(self.image_std))
        if getattr(self, "_video_geo", None) != geo:
            _lib.check(_lib.load().avh_set_video_preprocess(handle, H, W, geo[2], geo[3]))
            self._video_geo = geo

    @torch.no_grad()
    def extract_finetune_host(self, video, audio, padding_mask=None, output_layer=None, out=None, wait=True):
        """End-to-end call with HOST tensors (pinned recommended): H2D copies, forward and the D2H read of the
        features all happen inside ``avh_forward_host``.  video [B,1,T,88,88] (or raw uint8 [B,1,T,H,W]) / audio
        [B,F,T] CPU tensors (either may be None; made contiguous if they are not); returns a CPU tensor [B,T,D].
        ``wait=False`` only enqueues on the current stream (the caller synchronises it before reading ``out``),
        which lets several batches be in flight on different streams.  Same checks as ``extract_finetune``; the
        byte counts the library copies are those of the validated shapes."""
        self._check_mode(False)
        handle = self._ensure_handle()
        dev = self.encoder.layer_norm.weight.device
        video, video_dt, audio, pm, _, B, T = self._check_inputs(handle, video, audio, padding_mask, torch.device("cpu"))
        if audio is not None:
            audio = audio.contiguous()            # the host entry point reads a dense [B,F,T] block
        out_dtype = self.encoder.layer_norm.weight.dtype
        if out_dtype not in _DTYPES:
            out_dtype = torch.float32
        if out is None:
            out = torch.empty(B, T, self.encoder_embed_dim, dtype=out_dtype).pin_memory()
        elif (out.device.type != "cpu" or not out.is_contiguous() or out.dtype not in _DTYPES
              or tuple(out.shape) != (B, T, self.encoder_embed_dim)):
            raise ValueError(f"out must be a contiguous CPU tensor [{B},{T},{self.encoder_embed_dim}]")
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            lib = _lib.load()
            _lib.check((lib.avh_forward_host if wait else lib.avh_forward_host_async)(
                handle,
                ctypes.c_void_p(video.data_ptr()) if video is not None else None,
                video_dt,
                ctypes.c_void_p(audio.data_ptr()) if audio is not None else None,
                _DTYPES[audio.dtype] if audio is not None else 0,
                ctypes.c_void_p(pm.data_ptr()) if pm is not None else None,
                B, T, 0 if output_layer is None else int(output_layer),
                ctypes.c_void_p(out.data_ptr()), _DTYPES[out.dtype], ctypes.c_void_p(stream)))
            if not wait:
                # the async copy reads these host buffers after this call returns: keep them alive until the caller
                # has synchronised the stream (replaced by the next call on the same stream)
                self._host_keepalive[stream] = (video, audio, pm, out)
        return out

    def read_stage(self, name, numel):
        """Intermediate tensor of the last forward (needs cfg.capture_stages=True): 'resnet', 'fused_ln', 'enc_in'."""
        dev = self.encoder.layer_norm.weight.device
        dst = torch.empty(numel, device=dev, dtype=torch.float32)
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            _lib.check(_lib.load().avh_read_stage(self._handle, name.encode(), ctypes.c_void_p(dst.data_ptr()),
                                                  numel, ctypes.c_void_p(stream)))
        return dst

    def profile_forward(self, source, padding_mask=None, output_layer=None):
        """One forward with CUDA events around every launch; returns {class: {launches, ms, tc_flops}}."""
        import json
        handle = self._ensure_handle()
        lib = _lib.load()
        _lib.check(lib.avh_set_profiling(handle, 1))
        try:
            self.extract_finetune(source, padding_mask, output_layer=output_layer)
            buf = ctypes.create_string_buffer(1 << 16)
            _lib.check(lib.avh_profile_json(handle, buf, len(buf)))
        finally:
            lib.avh_set_profiling(handle, 0)
        return json.loads(buf.value.decode())

    # ------------------------------------------------------------------ pretraining-mode extras (SURVEY 8(f) rank 4)
    def _substitute(self, x, layout, B, T, U, codes, emb, channel_zero=None):
        """avh_mask_substitute on a device tensor: layout 0 = contiguous [B,T,U] units, 1 = strided [B,U,T]."""
        dev = x.device
        if dev.type != "cuda":
            raise RuntimeError("span masking runs on the device: move the inputs to the module's CUDA device")
        if x.dtype not in _DTYPES:
            raise ValueError(f"unsupported dtype {x.dtype}")
        code_dev = torch.from_numpy(np.ascontiguousarray(codes, dtype=np.int32)).to(dev)
        out = torch.empty(x.shape, device=dev, dtype=x.dtype)
        strides = (ctypes.c_int64 * 3)(*x.stride()) if layout == 1 else None
        if layout == 0:
            x = x.contiguous()
        emb_t = emb.detach().to(dev).contiguous() if emb is not None else None
        cz = channel_zero.to(device=dev, dtype=torch.bool).contiguous().view(torch.uint8) if channel_zero is not None else None
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            _lib.check(_lib.load().avh_mask_substitute(
                ctypes.c_void_p(x.data_ptr()), _DTYPES[x.dtype], layout, strides, B, T, U,
                ctypes.c_void_p(code_dev.data_ptr()),
                ctypes.c_void_p(emb_t.data_ptr()) if emb_t is not None else None,
                _DTYPES[emb_t.dtype] if emb_t is not None else 0,
                ctypes.c_void_p(cz.data_ptr()) if cz is not None else None,
                ctypes.c_void_p(out.data_ptr()), _DTYPES[out.dtype], ctypes.c_void_p(stream)))
        return out

    @torch.no_grad()
    def apply_input_mask(self, x, padding_mask, target_list=None):
        """avhubert/hubert.py:442-494.  x = audio [B,F,T] or video [B,1,T,H,W] on the device.  The spans come from
        masking.compute_mask_indices (numpy's global generator, the reference's draw order); masked audio frames
        become ``mask_emb``, masked video frames the same frames of another clip ('same_other_seq': the shift drawn
        with torch.randint as the reference does) or another run of the same clip ('same_seq'); zeros when B == 1.
        Returns (a new contiguous tensor, mask_indices bool [B,T] on the device) — (x, None) when the probability is 0."""
        if x is None:
            raise ValueError("apply_input_mask needs both modalities (the reference fails on None, hubert.py:443)")
        c = self.cfg
        B, C, T = x.shape[:3]
        is_audio = x.dim() == 3
        prob, length = (c.mask_prob_audio, c.mask_length_audio) if is_audio else (c.mask_prob_image, c.mask_length_image)
        if not prob > 0:
            return x, None
        if not is_audio and (x.dim() != 5 or C != 1):
            raise ValueError(f"video must be [B,1,T,H,W], got {tuple(x.shape)}")
        m, starts, ends, owners = masking.compute_mask_indices(
            (B, T), padding_mask, prob, length, c.mask_selection, c.mask_other, min_masks=2,
            no_overlap=c.no_mask_overlap, min_space=c.mask_min_space)
        if B == 1:
            codes = masking.span_codes_constant(m, masking.ZERO)
        elif is_audio:
            codes = masking.span_codes_constant(m, masking.EMB)
        elif c.selection_type == "same_other_seq":
            perm = (torch.arange(B) + torch.randint(low=1, high=B, size=(1,))) % B
            codes = masking.span_codes_other_clip(m, perm.numpy())
        elif c.selection_type == "same_seq":
            codes = masking.span_codes_same_clip(m, starts, ends, owners)
        else:
            raise ValueError(f"unknown selection_type {c.selection_type}")
        if is_audio:
            out = self._substitute(x, 1, B, T, C, codes, self.mask_emb)
        else:
            out = self._substitute(x, 0, B, T, x.size(3) * x.size(4), codes, None)
        return out, torch.from_numpy(m).to(x.device)

    @torch.no_grad()
    def apply_feature_mask(self, x, padding_mask, target_list=None):
        """avhubert/hubert.py:496-536 on token rows x [B,T,D]: masked rows become ``mask_emb``; with mask_channel_prob
        > 0 whole channels of a clip are zeroed.  Returns (new tensor, mask_indices or None)."""
        c = self.cfg
        B, T, C = x.shape
        if c.mask_prob_audio != c.mask_prob_image or c.mask_length_audio != c.mask_length_image:
            raise AssertionError("masking prob/length for image/audio be same for feature masking")
        m = None
        codes = np.full((B, T), masking.KEEP, dtype=np.int32)
        if c.mask_prob_audio > 0:
            m, _, _, _ = masking.compute_mask_indices(
                (B, T), padding_mask, c.mask_prob_audio, c.mask_length_image, c.mask_selection, c.mask_other,
                min_masks=2, no_overlap=c.no_mask_overlap, min_space=c.mask_min_space)
            codes = masking.span_codes_constant(m, masking.EMB)
        cz = None
        if c.mask_channel_prob > 0:
            mc, _, _, _ = masking.compute_mask_indices(
                (B, C), None, c.mask_channel_prob, c.mask_channel_length, c.mask_channel_selection,
                c.mask_channel_other, no_overlap=c.no_mask_channel_overlap, min_space=c.mask_channel_min_space)
            cz = torch.from_numpy(mc)
        out = self._substitute(x, 0, B, T, C, codes, self.mask_emb, cz)
        return out, (torch.from_numpy(m).to(x.device) if m is not None else None)

    @torch.no_grad()
    def compute_logits(self, feats, emb_mat, bias=None, sim_type=None, logit_temp=None):
        """avhubert/hubert.py:576-589: feats [B,T,F] (or [M,F]), emb_mat [V,F] -> fp32 logits [B,T,V]; cosine or dot
        similarity over the last dim divided by ``logit_temp``.  (``bias`` turns the 'dot' form into nn.Linear.)"""
        sim_type = self.cfg.sim_type if sim_type is None else sim_type
        if sim_type not in ("dot", "cosine"):
            raise NotImplementedError
        temp = float(self.cfg.logit_temp if logit_temp is None else logit_temp)
        dev = feats.device
        if dev.type != "cuda":
            raise RuntimeError("compute_logits runs on the device (there is no CPU path)")
        lead, K = feats.shape[:-1], feats.size(-1)
        f2 = feats.reshape(-1, K)
        if f2.dtype not in _DTYPES or f2.stride(-1) != 1:
            f2 = f2.float().contiguous()
        e2 = emb_mat.detach()
        if e2.dtype not in _DTYPES or e2.stride(-1) != 1 or e2.device != dev:
            e2 = e2.to(dev).float().contiguous()
        if e2.dim() != 2 or e2.size(1) != K:
            raise ValueError(f"emb_mat must be [V,{K}], got {tuple(emb_mat.shape)}")
        b = bias.detach().to(dev).float().contiguous() if bias is not None else None
        M, V = f2.size(0), e2.size(0)
        out = torch.empty(M, V, device=dev, dtype=torch.float32)
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            _lib.check(_lib.load().avh_compute_logits(
                ctypes.c_void_p(f2.data_ptr()), _DTYPES[f2.dtype], f2.stride(0) if M > 1 else K,
                ctypes.c_void_p(e2.data_ptr()), _DTYPES[e2.dtype], e2.stride(0) if V > 1 else K,
                ctypes.c_void_p(b.data_ptr()) if b is not None else None, M, V, K,
                1 if sim_type == "cosine" else 0, temp, ctypes.c_void_p(out.data_ptr()), V, ctypes.c_void_p(stream)))
        return out.view(*lead, V)

    def _features_pen(self, numel):
        """features.float().pow(2).mean() over the fused (pre-LayerNorm) features of the last forward (hubert.py:629)."""
        dev = self.encoder.layer_norm.weight.device
        stage = self.read_stage("fused", numel)
        acc = torch.zeros(1, device=dev, dtype=torch.float64)
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            _lib.check(_lib.load().avh_sum_squares(ctypes.c_void_p(stage.data_ptr()), _lib.AVH_F32, numel,
                                                  ctypes.c_void_p(acc.data_ptr()), ctypes.c_void_p(stream)))
        return (acc / numel).float().squeeze(0)

    def _need_stages(self):
        if not self.cfg.capture_stages:           # the encoder input is only kept when the handle captures stages
            self.cfg.capture_stages = True
            self._destroy_handle()
            self._dirty = True

    @torch.no_grad()
    def extract_features(self, source, padding_mask=None, mask=False, ret_conv=False, output_layer=None):
        """avhubert/hubert.py:676-692 (forward(features_only=True), :591-653) in eval mode: returns
        (features [B,T,D], padding_mask).  ``ret_conv=True`` gives the encoder INPUT (post_extract_proj output with
        padded frames zeroed, as the reference's in-place index_put leaves it) — layer 0 of
        avhubert/clustering/dump_hubert_feature.py:95-106; otherwise the output of layer ``output_layer`` (1-based,
        no final LayerNorm) or of the whole encoder.  Both modalities are required, as in the reference."""
        res = self.forward(source, padding_mask=padding_mask, mask=mask, features_only=True, output_layer=output_layer,
                           _want_features=ret_conv)
        return (res["features"] if ret_conv else res["x"]), res["padding_mask"]

    @torch.no_grad()
    def forward(self, source, target_list=None, padding_mask=None, mask=True, features_only=False, output_layer=None,
                _want_features=True):
        """The masked-prediction forward, avhubert/hubert.py:591-674, in EVAL mode (what fairseq's validation step and
        ``extract_features`` run; the training-mode pass needs the backward of SURVEY row A18).  Input span masking
        (``masking_type='input'``: frames substituted before the frontends) or feature masking (``'feature'``: token
        rows replaced by ``mask_emb`` after post_extract_proj), the encoder, then — unless ``features_only`` —
        final_proj, cosine / dot logits against the label embeddings and the masked / unmasked selections.  Returns
        the reference's dict.  numpy / torch CPU generators are consumed in the reference's order."""
        if self.training:
            raise NotImplementedError("the pretraining forward runs in eval mode here (modality dropout and the "
                                      "losses' backward belong to the training configuration, SURVEY row A18)")
        src_audio, src_video = source["audio"], source["video"]
        if src_audio is None or src_video is None:
            raise ValueError("forward / extract_features need both modalities (forward_features fails on None in the "
                             "reference, hubert.py:609-610); use extract_finetune for single-modality input")
        c = self.cfg
        mask_indices = None
        if mask and c.masking_type == "input":
            src_video, mi_v = self.apply_input_mask(src_video, padding_mask, target_list)
            src_audio, mi_a = self.apply_input_mask(src_audio, padding_mask, target_list)
            mask_indices = torch.logical_or(mi_a, mi_v)      # None here fails as in the reference (prob 0 + mask=True)
        np.random.random(), np.random.random()               # modality-dropout coins: drawn in eval mode too (:611)
        if target_list is not None:
            T = src_video.size(2)
            if self.feat2tar_ratio * T > min(t.size(1) for t in target_list):
                raise NotImplementedError("labels shorter than the features (forward_targets would trim the features "
                                          "mid-forward, hubert.py:553-558): trim the inputs to the labelled frames")
            idx = (torch.arange(T).float() * self.feat2tar_ratio).long()
            target_list = [t[:, idx.to(t.device)] for t in target_list]
        feature_mask = bool(mask) and c.masking_type == "feature"
        want_pen = not features_only
        if _want_features or feature_mask or want_pen:
            self._need_stages()
        src = {"audio": src_audio, "video": src_video}
        if not feature_mask:
            x, pm = self.extract_finetune(src, padding_mask, output_layer=output_layer)
            B, T, D = x.shape
            features = None
            if _want_features:
                features = self.read_stage("enc_in", B * T * D).view(B, T, D).to(x.dtype)
        else:
            # features after post_extract_proj (one encoder layer is computed and discarded), mask rows, run the encoder
            y1, pm = self.extract_finetune(src, padding_mask, output_layer=1)
            B, T, D = y1.shape
            feats = self.read_stage("enc_in", B * T * D).view(B, T, D).to(y1.dtype)
            pen = self._features_pen(B * T * self.embed) if want_pen else None
            features, mask_indices = self.apply_feature_mask(feats, pm, target_list)
            x = self._encoder_forward(features, pm, output_layer)
        if features_only:
            return {"x": x, "padding_mask": pm, "features": features}
        if not feature_mask:
            pen = self._features_pen(B * T * self.embed)
        if self.final_proj is None or self.num_classes is None:
            raise RuntimeError("the masked-prediction head was removed (remove_pretraining_modules) or the model was "
                               "built without dictionaries")
        label_embs_list = self.label_embs_concat.split(self.num_classes, 0)
        proj_x = self.compute_logits(x, self.final_proj.weight, bias=self.final_proj.bias, sim_type="dot", logit_temp=1.0)
        if self.untie_final_proj:
            proj_x_list = proj_x.chunk(len(self.num_classes), dim=-1)
        else:
            proj_x_list = [proj_x for _ in self.num_classes]
        logit_list = [self.compute_logits(p, e).view(-1, n) for p, e, n in zip(proj_x_list, label_embs_list, self.num_classes)]
        if pm is None:       # the reference evaluates ~padding_mask here (hubert.py:663)
            raise TypeError("forward(features_only=False) needs a padding_mask (bad operand type for unary ~: 'NoneType')")
        pad = pm
        sel_m = torch.logical_and(mask_indices, ~pad).view(-1)
        sel_u = torch.logical_and(~mask_indices, ~pad).view(-1)
        return {
            "logit_m_list": [lg[sel_m] for lg in logit_list],
            "logit_u_list": [lg[sel_u] for lg in logit_list],
            "target_m_list": [t.reshape(-1).to(x.device)[sel_m].long() for t in target_list],
            "target_u_list": [t.reshape(-1).to(x.device)[sel_u].long() for t in target_list],
            "padding_mask": pm,
            "features_pen": pen,
        }

    def _encoder_forward(self, feats, padding_mask, output_layer):
        """self.encoder(x, padding_mask, layer) on caller features through avh_encoder_forward."""
        dev = feats.device
        B, T, D = feats.shape
        feats = feats.contiguous()
        out = torch.empty(B, T, D, device=dev, dtype=feats.dtype)
        pm_u8 = padding_mask.to(device=dev, dtype=torch.bool).contiguous().view(torch.uint8) if padding_mask is not None else None
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            _lib.check(_lib.load().avh_encoder_forward(
                self._ensure_handle(), ctypes.c_void_p(feats.data_ptr()), _DTYPES[feats.dtype],
                ctypes.c_void_p(pm_u8.data_ptr()) if pm_u8 is not None else None, B, T,
                0 if output_layer is None else int(output_layer), ctypes.c_void_p(out.data_ptr()), _DTYPES[out.dtype],
                ctypes.c_void_p(stream)))
        return out
