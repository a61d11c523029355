"""Host side of the device backward shared by the three autograd wrappers (TransformerEncoder, the fusion tail, the whole
AVHubertModel): one call into the library that fills a flat gradient buffer in the parameters' dtype bucket by bucket,
and — when a GradientAllReducer is attached to the module — the all-reduce of every bucket issued on a side stream as
soon as the library has recorded the bucket's event, so that the collective overlaps the rest of the backward
(fairseq legacy_distributed_data_parallel.py:76-165 does the reduction after the backward; same result)."""
import ctypes
import itertools

import numpy as np
import torch

from . import _lib

_DTYPES = {torch.float32: _lib.AVH_F32, torch.float16: _lib.AVH_F16, torch.bfloat16: _lib.AVH_BF16}
PARAMS_PER_LAYER = 16      # gradient tensors of one encoder layer, first in every training step's parameter list


class StepRegularization:
    """Dropout and LayerDrop of one training step (avh_set_train_args).  The LayerDrop coins are drawn here, one
    np.random.random() per layer in layer order, as the reference draws them (wav2vec2.py:886-888) whatever the
    probability; the dropout seed comes from torch's CPU generator, and only when some dropout probability is non-zero."""

    def __init__(self, n_layers, dropout_input=0.0, dropout=0.0, activation_dropout=0.0, attention_dropout=0.0,
                 layerdrop=0.0):
        if float(attention_dropout or 0.0) != 0.0:
            raise NotImplementedError("attention_dropout > 0 in training mode is not implemented (0.0 in every "
                                      "shipped fine-tune config, avhubert/conf/finetune/*.yaml)")
        self.p = (float(dropout_input or 0.0), float(dropout or 0.0), float(activation_dropout or 0.0))
        self.layerdrop = float(layerdrop or 0.0)
        self.skip = [0 if np.random.random() > self.layerdrop else 1 for _ in range(n_layers)]
        if self.layerdrop <= 0.0:
            self.skip = [0] * n_layers
        self.seed = int(torch.randint(0, 2 ** 62, (1,)).item()) if any(p > 0.0 for p in self.p) else 0

    def set_on(self, handle):
        """Leaves the regularisation for the next training forward on `handle`."""
        skip = (ctypes.c_uint8 * len(self.skip))(*self.skip) if self.layerdrop > 0.0 else None
        ta = _lib.AvhTrainArgs(dropout_input=self.p[0], dropout=self.p[1], activation_dropout=self.p[2], attention_dropout=0.0,
                               bn_momentum=0.1, seed=self.seed,
                               layer_skip=ctypes.cast(skip, ctypes.c_void_p) if skip is not None else None)
        _lib.check(_lib.load().avh_set_train_args(handle, ctypes.byref(ta)))

    def layer_grads(self, grads, reduced):
        """autograd's view of a dropped layer: its parameters took no part in the step, so their gradients are None —
        unless the all-reducer has reduced the bucket, whose values (the other ranks' gradients) they then get."""
        if reduced:
            return grads
        grads = list(grads)
        for l, dropped in enumerate(self.skip):
            if dropped:
                grads[l * PARAMS_PER_LAYER:(l + 1) * PARAMS_PER_LAYER] = [None] * PARAMS_PER_LAYER
        return grads


def backward_flat(handle, dout, dx, n_floats, dtypes, fwd_stream, owner):
    """Runs the library backward of the last training forward on `handle`.  Returns {dtype: flat gradient buffer}: when
    every parameter has the same dtype the buffer is written in that dtype directly (and all-reduced bucket by bucket if
    `owner._grad_sync` is an active GradientAllReducer); otherwise fp32, converted once per dtype on demand."""
    dev = dout.device
    lib = _lib.load()
    vp = ctypes.c_void_p
    single = dtypes[0] if dtypes and all(d == dtypes[0] for d in dtypes) and dtypes[0] in _DTYPES else None
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        if stream != fwd_stream:
            raise RuntimeError("the backward must run on the CUDA stream of its forward")
        dxp = vp(dx.data_ptr()) if dx is not None else None
        dxd = _DTYPES[dx.dtype] if dx is not None else 0
        if single is None:
            flat = torch.empty(n_floats, device=dev, dtype=torch.float32)
            _lib.check(lib.avh_encoder_backward(handle, vp(dout.data_ptr()), _DTYPES[dout.dtype], dxp, dxd, vp(flat.data_ptr()),
                                                n_floats, vp(stream)))
            return _FlatGrads(flat)
        flat = torch.empty(n_floats, device=dev, dtype=single)
        _lib.check(lib.avh_encoder_backward_buckets(handle, vp(dout.data_ptr()), _DTYPES[dout.dtype], dxp, dxd,
                                                    vp(flat.data_ptr()), _DTYPES[single], n_floats, vp(stream)))
        sync = getattr(owner, "_grad_sync", None)
        reduced = sync is not None and sync.reduce_buckets(lib, handle, flat)
    out = _FlatGrads(flat)
    out.reduced = bool(reduced)
    return out


class _FlatGrads:
    """The flat buffer in one dtype, other dtypes converted once on demand."""

    def __init__(self, flat):
        self.base = flat
        self.by_dtype = {flat.dtype: flat}
        self.reduced = False

    def of(self, dt):
        if dt not in self.by_dtype:
            self.by_dtype[dt] = self.base.to(dt)
        return self.by_dtype[dt]


def refresh_weights_device(handle, module, prefix=""):
    """After an optimizer step: rewrite the packed weights the training plans read from `module`'s device-resident
    parameters, in place and on the device (avh_refresh_weights_device) — plans and captured graphs stay valid, nothing
    crosses the host.  `prefix` maps the module's parameter names onto the state-dict keys the handle was loaded with."""
    _refresh(handle, "avh_refresh_weights_device", module.named_parameters(), prefix)


def refresh_eval_weights_device(handle, module, prefix=""):
    """Before an eval forward that follows training: the same refresh on a trainable handle, then the eval-only packed
    forms (BatchNorm folded with the running statistics, the conv2 + shortcut GEMM weights) from `module`'s parameters
    and buffers, in place on the device (avh_refresh_eval_weights_device), bit-identical to a full re-pack."""
    _refresh(handle, "avh_refresh_eval_weights_device", itertools.chain(module.named_parameters(), module.named_buffers()),
             prefix)


def _refresh(handle, entry, named_tensors, prefix):
    lib = _lib.load()
    names, tensors = [], []
    for name, p in named_tensors:
        t = p.detach()
        if not t.is_floating_point():
            continue
        if t.dtype not in _DTYPES:
            t = t.float()
        names.append((prefix + name).encode())
        tensors.append(t.contiguous())
    n = len(names)
    c_names = (ctypes.c_char_p * n)(*names)
    c_ptrs = (ctypes.c_void_p * n)(*[t.data_ptr() for t in tensors])
    c_dts = (ctypes.c_int32 * n)(*[_DTYPES[t.dtype] for t in tensors])
    c_num = (ctypes.c_int64 * n)(*[t.numel() for t in tensors])
    dev = tensors[0].device
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        _lib.check(getattr(lib, entry)(handle, c_names, c_ptrs, c_dts, c_num, n, ctypes.c_void_p(stream)))
