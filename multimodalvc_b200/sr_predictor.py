"""Mirrors of two users of fairseq's wav2vec2 ``TransformerEncoder`` outside AV-HuBERT itself (SURVEY 8(f)-4):

* ``TransformerEncoder`` — ``fairseq/fairseq/models/wav2vec/wav2vec2.py:816-902`` as a parameter container whose
  ``forward(x, padding_mask=None, layer=None)`` runs in ``libavh_b200.so`` (``avh_encoder_forward``: positional conv +
  GELU, pre-/post-LN layers with the tcgen05 GEMMs and attention kernels of the AV-HuBERT path, final LayerNorm);
* ``Speech_Rate_Predictor`` — ``src/sub_model/modules.py:108-142``: ``Linear(1024, 256)`` on the Whisper features, a
  learned ``sr_token`` prepended, a 2-layer ``TransformerEncoder`` (d = 256, 4 heads, FFN 1024), ``Linear(256, 1)`` +
  ReLU on the token's output.  Same attribute / state-dict names as the reference (``sr_token``, ``linear.*``,
  ``encoder.*``, ``sr_predictor.*``).

Inference by default (eval mode: LayerDrop and dropout are identity, as in the reference's ``self.training`` gates).
``TransformerEncoder(args, trainable=True)`` also differentiates: in ``.train()`` with gradients enabled ``forward`` is a
``torch.autograd.Function`` whose backward is the library's (``avh_encoder_train_forward`` / ``avh_encoder_backward``:
SURVEY row A18, encoder part of BASELINE config 5; pre-LN and post-LN layers; ``dropout``, ``activation_dropout`` and
``encoder_layerdrop`` of the args as the reference applies them, ``attention_dropout`` must be 0), so ``loss.backward()``
fills ``.grad`` of the input and of every encoder parameter (None for the layers LayerDrop dropped).  No CPU path.
"""
import ctypes
from types import SimpleNamespace

import torch
import torch.nn as nn

from . import _lib
from ._train import StepRegularization, backward_flat, refresh_weights_device
from .hubert import _DTYPES, _EncoderParams
from .hubert_asr import _project


class _EncoderTrainFn(torch.autograd.Function):
    """y = encoder(x, padding_mask) with the library's forward (activations saved in the handle's plan) and backward.
    The parameters are passed only so that autograd routes their gradients; the arithmetic uses the packed copies."""

    @staticmethod
    def forward(ctx, enc, reg, x, pm_u8, *params):
        handle = enc._ensure_handle()
        dev = x.device
        B, T, D = x.shape
        out_dtype = enc.layer_norm.weight.dtype if enc.layer_norm.weight.dtype in _DTYPES else torch.float32
        out = torch.empty(B, T, D, device=dev, dtype=out_dtype)
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            reg.set_on(handle)
            _lib.check(_lib.load().avh_encoder_train_forward(
                handle, ctypes.c_void_p(x.data_ptr()), _DTYPES[x.dtype],
                ctypes.c_void_p(pm_u8.data_ptr()) if pm_u8 is not None else None, B, T,
                ctypes.c_void_p(out.data_ptr()), _DTYPES[out_dtype], ctypes.c_void_p(stream)))
        ctx.enc, ctx.reg, ctx.handle, ctx.x_dtype, ctx.stream = enc, reg, handle, x.dtype, stream
        ctx.shapes = [tuple(p.shape) for p in params]
        ctx.dtypes = [p.dtype for p in params]
        ctx.params = params
        return out

    @staticmethod
    def backward(ctx, dout):
        enc = ctx.enc
        dev = dout.device
        dout = dout.contiguous()
        if dout.dtype not in _DTYPES:
            dout = dout.float()
        lib = _lib.load()
        n = ctypes.c_int64()
        _lib.check(lib.avh_encoder_grad_count(ctx.handle, ctypes.byref(n)))
        dx = torch.empty(dout.shape, device=dev, dtype=ctx.x_dtype)
        flat = backward_flat(ctx.handle, dout, dx, n.value, ctx.dtypes, ctx.stream, enc)
        grads, off = [], 0
        for shape, dt in zip(ctx.shapes, ctx.dtypes):
            k = 1
            for d in shape:
                k *= d
            grads.append(flat.of(dt)[off:off + k].view(shape))
            off += k
        assert off == n.value
        if flat.reduced:
            enc._grad_sync.mark_reduced(ctx.params)
        return (None, None, dx, None, *ctx.reg.layer_grads(grads, flat.reduced))


class TransformerEncoder(nn.Module):
    """``TransformerEncoder(args)`` with the reference's argument names (encoder_embed_dim, encoder_ffn_embed_dim,
    encoder_attention_heads, encoder_layers, conv_pos, conv_pos_groups, layer_norm_first, activation_fn='gelu')."""

    def __init__(self, args, trainable=False):
        super().__init__()
        self.trainable = bool(trainable)
        if getattr(args, "activation_fn", "gelu") != "gelu":
            raise NotImplementedError("only activation_fn='gelu' is implemented")
        if args.encoder_embed_dim != 64 * args.encoder_attention_heads:
            raise NotImplementedError("the attention kernels need head_dim 64")
        self.args = args
        p = _EncoderParams(SimpleNamespace(
            encoder_embed_dim=args.encoder_embed_dim, encoder_ffn_embed_dim=args.encoder_ffn_embed_dim,
            encoder_layers=args.encoder_layers, conv_pos=args.conv_pos, conv_pos_groups=args.conv_pos_groups,
            layer_norm_first=args.layer_norm_first))
        self.embedding_dim = p.embedding_dim
        self.layer_norm_first = p.layer_norm_first
        self.pos_conv, self.layers, self.layer_norm = p.pos_conv, p.layers, p.layer_norm
        self._handle, self._handle_key, self._dirty = None, None, True
        self.register_load_state_dict_post_hook(lambda module, incompatible: module._mark_dirty())

    def _mark_dirty(self):
        self._dirty = True

    def _apply(self, fn, *a, **k):
        out = super()._apply(fn, *a, **k)
        self._dirty = True
        return out

    def refresh_weights(self):
        self._dirty = True

    def __del__(self):
        try:
            if self._handle is not None:
                _lib.load().avh_destroy(self._handle)
        except Exception:
            pass

    def _ensure_handle(self):
        p = self.layer_norm.weight
        if p.device.type != "cuda":
            raise RuntimeError("multimodalvc_b200.TransformerEncoder computes on a B200 only (there is no CPU path)")
        mode = _lib.AVH_COMPUTE_FP32 if p.dtype == torch.float32 else _lib.AVH_COMPUTE_BF16
        key = (p.device.index if p.device.index is not None else torch.cuda.current_device(), mode)
        if not self.training and getattr(self, "_eval_stale", False):
            self._dirty, self._eval_stale = True, False      # the device-side refresh skipped the eval-only packed forms
        if self._handle is not None and key == self._handle_key and not self._dirty:
            return self._handle
        lib = _lib.load()
        if self._handle is None or key != self._handle_key:
            if self._handle is not None:
                lib.avh_destroy(self._handle)
            a = self.args
            cc = _lib.AvhConfig(
                encoder_layers=a.encoder_layers, encoder_embed_dim=a.encoder_embed_dim,
                encoder_ffn_embed_dim=a.encoder_ffn_embed_dim, encoder_attention_heads=a.encoder_attention_heads,
                audio_feat_dim=0, modality_fuse=_lib.AVH_FUSE_ADD, layer_norm_first=int(bool(a.layer_norm_first)),
                conv_pos=a.conv_pos, conv_pos_groups=a.conv_pos_groups, compute_mode=mode, frontend_chunk_frames=0,
                capture_stages=0)
            cc.reserved[0] = 1                    # bare TransformerEncoder: only "encoder.*" weights
            cc.reserved[3] = 1 if self.trainable else 0      # also pack the backward's transposed operands
            hp = ctypes.c_void_p()
            _lib.check(lib.avh_create(ctypes.byref(cc), key[0], ctypes.byref(hp)))
            self._handle, self._handle_key = hp, key
        with torch.no_grad():
            for name, t in self.state_dict().items():
                t = t.detach().contiguous()
                if t.dtype not in _DTYPES:
                    t = t.float()
                shape = (ctypes.c_int64 * max(t.dim(), 1))(*t.shape)
                _lib.check(lib.avh_load_tensor(self._handle, ("encoder." + name).encode(), ctypes.c_void_p(t.data_ptr()),
                                               _DTYPES[t.dtype], shape, t.dim()))
            torch.cuda.synchronize(p.device)
        _lib.check(lib.avh_finalize_weights(self._handle))
        _lib.check(lib.avh_drop_host_weights(self._handle))
        self._dirty = False
        return self._handle

    def grad_parameters(self):
        """The parameters in the order avh_encoder_backward writes their gradients (include/avh_b200.h)."""
        out = []
        for layer in self.layers:
            a = layer.self_attn
            out += [a.q_proj.weight, a.k_proj.weight, a.v_proj.weight, a.q_proj.bias, a.k_proj.bias, a.v_proj.bias,
                    a.out_proj.weight, a.out_proj.bias, layer.self_attn_layer_norm.weight, layer.self_attn_layer_norm.bias,
                    layer.fc1.weight, layer.fc1.bias, layer.fc2.weight, layer.fc2.bias,
                    layer.final_layer_norm.weight, layer.final_layer_norm.bias]
        out += [self.layer_norm.weight, self.layer_norm.bias]
        pc = self.pos_conv[0]
        out += [pc.bias, pc.weight_g, pc.weight_v]
        return out

    def _forward_train(self, x, padding_mask, layer):
        a = self.args
        if not self.trainable:
            raise RuntimeError("build the module with trainable=True to differentiate through it (or call .eval())")
        if layer is not None:
            raise NotImplementedError("the training-mode forward runs the whole stack (layer=None)")
        dev = self.layer_norm.weight.device
        if x.device != dev or x.dim() != 3 or x.size(2) != self.embedding_dim:
            raise ValueError(f"x must be [B,T,{self.embedding_dim}] on {dev}, got {tuple(x.shape)} on {x.device}")
        B, T, _ = x.shape
        if x.dtype not in _DTYPES:
            x = x.float()
        x = x.contiguous()
        pm = None
        if padding_mask is not None:
            if tuple(padding_mask.shape) != (B, T):
                raise ValueError(f"padding_mask must be [{B},{T}]")
            pm = padding_mask.to(device=dev, dtype=torch.bool).contiguous().view(torch.uint8)
        if not hasattr(self, "_versions"):
            self._dirty = True
        elif any(p._version != v for p, v in zip(self.parameters(), self._versions)):
            if self._handle is not None and not self._dirty:     # an optimizer step changed the weights: refresh the packed
                refresh_weights_device(self._handle, self, "encoder.")   # copies in place on the device (eval forms go stale)
                self._eval_stale = True
            else:
                self._dirty = True
        reg = StepRegularization(a.encoder_layers, dropout=getattr(a, "dropout", 0.0),
                                 activation_dropout=getattr(a, "activation_dropout", 0.0),
                                 attention_dropout=getattr(a, "attention_dropout", 0.0),
                                 layerdrop=getattr(a, "encoder_layerdrop", 0.0))
        self._ensure_handle()
        self._versions = [p._version for p in self.parameters()]
        y = _EncoderTrainFn.apply(self, reg, x, pm, *self.grad_parameters())
        self._last_train_args = (reg.seed, list(reg.skip))      # what the step used: tests rebuild its masks from it
        return y, []

    def forward(self, x, padding_mask=None, layer=None):
        """wav2vec2.py:859-902: returns (x [B,T,D], layer_results) — layer_results is empty (nobody on this path reads
        it; the reference fills it with per-layer tensors only for tgt_layer / feature dumping)."""
        if self.training and torch.is_grad_enabled():
            return self._forward_train(x, padding_mask, layer)
        with torch.no_grad():
            return self._forward_eval(x, padding_mask, layer)

    def _forward_eval(self, x, padding_mask=None, layer=None):
        if self.training and not self.trainable:
            raise RuntimeError("TransformerEncoder on the device path is inference-only: call .eval()")
        handle = self._ensure_handle()
        dev = self.layer_norm.weight.device
        if x.device != dev or x.dim() != 3 or x.size(2) != self.embedding_dim:
            raise ValueError(f"x must be [B,T,{self.embedding_dim}] on {dev}, got {tuple(x.shape)} on {x.device}")
        B, T, D = x.shape
        if B < 1 or T < 1:
            raise ValueError("empty batch")
        if x.dtype not in _DTYPES:
            x = x.float()
        x = x.contiguous()
        pm = None
        if padding_mask is not None:
            if tuple(padding_mask.shape) != (B, T):
                raise ValueError(f"padding_mask must be [{B},{T}]")
            pm = padding_mask.to(device=dev, dtype=torch.bool).contiguous().view(torch.uint8)
        out_dtype = self.layer_norm.weight.dtype if self.layer_norm.weight.dtype in _DTYPES else torch.float32
        out = torch.empty(B, T, D, device=dev, dtype=out_dtype)
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            _lib.check(_lib.load().avh_encoder_forward(
                handle, ctypes.c_void_p(x.data_ptr()), _DTYPES[x.dtype],
                ctypes.c_void_p(pm.data_ptr()) if pm is not None else None, B, T,
                0 if layer is None else int(layer) + 1,       # fairseq's tgt_layer is 0-based (wav2vec2.py:892-894)
                ctypes.c_void_p(out.data_ptr()), _DTYPES[out_dtype], ctypes.c_void_p(stream)))
        return out, []


class Speech_Rate_Predictor(nn.Module):
    """src/sub_model/modules.py:108-142."""

    def __init__(self, num_layers):
        super().__init__()
        args = SimpleNamespace(dropout=0.0, encoder_embed_dim=256, conv_pos=128, conv_pos_groups=16,
                               encoder_ffn_embed_dim=1024, encoder_attention_heads=4, attention_dropout=0.0,
                               activation_dropout=0.1, activation_fn="gelu", layer_norm_first=True,
                               encoder_layers=num_layers, encoder_layerdrop=0.1)
        self.sr_token = nn.Parameter(torch.zeros(1, 1, 256))
        nn.init.xavier_uniform_(self.sr_token)
        self.linear = nn.Linear(1024, 256)
        self.encoder = TransformerEncoder(args)
        self.sr_predictor = nn.Linear(256, 1)
        self.activation = nn.ReLU()

    @torch.no_grad()
    def forward(self, x):
        """x [B,T,1024] (Whisper encoder features) -> speech-rate prediction [B,1]."""
        if self.training:
            raise RuntimeError("Speech_Rate_Predictor on the device path is inference-only: call .eval()")
        x = _project(x, self.linear)                                   # [B,T,256] on the tcgen05 GEMM
        tok = self.sr_token.to(x.dtype).expand(x.size(0), -1, -1)
        x = torch.cat([tok, x], dim=1)
        x, _ = self.encoder(x)
        return self.activation(_project(x[:, :1, :].contiguous(), self.sr_predictor)[:, 0, :])
