"""SpectralConv / SpectralAttention -- drop-in for `makani.models.common.{SpectralConv, SpectralAttention}`
(/root/reference/makani/models/common/spectral_convolution.py:37-264 and :267-519) on top of the CUDA library.

Same constructor signatures, parameter names / shapes / dtypes (`weight` complex64 [G, Cin/G, Cout/G, L(, M)], `bias`
[1, Cout, 1, 1]; `w`, `wout`, `b`, `activations`), the `is_shared_mp` / `sharded_dims_mp` tags the reference's DDP hook
and flexible checkpoints read (spectral_convolution.py:195-203,210-211), the same ValueErrors, and `forward(x) -> (y, residual)`.

The whole forward is 5 kernels: longitude FFT -> Legendre analysis -> channel mix -> Legendre synthesis -> inverse FFT
(+bias, +cast); the spectral tensors stay in the packed layout between them.
"""
import ctypes
import math
import warnings

import weakref

import torch
import torch.nn as nn

from . import _lib
from ._lib import B200ShtError
from .sht import RealSHT, InverseRealSHT, _ptr, _stream, resolve_precision, _SpecPack, _SpecUnpack

_VP = ctypes.c_void_p

_DENSE_OPS = (_lib.OP_DHCONV, _lib.OP_SHARED, _lib.OP_LDEP)


def _op_code(operator_type, separable):
    if operator_type == "dhconv":
        return _lib.OP_SEP_DHCONV if separable else _lib.OP_DHCONV
    if operator_type == "diagonal":
        return _lib.OP_SEP_DIAGONAL if separable else _lib.OP_DIAGONAL
    raise ValueError(f"Unknown operator type {operator_type}")


_warned_mix_fallback = set()


def mix_pack_precision(op, B, G, Ci, Co, precision):
    """Precision the packed weight must be prepared for.  The tcgen05 channel mix (precision tf32) needs a batch that divides 32 and
    16-byte aligned group slices; other shapes are served by the fp32 CUDA-core kernels (correct, slower).  In that case the weight is NOT
    rounded to TF32 (the result is then plain fp32, not a mixture) and the user is told once per shape."""
    if precision != _lib.PREC_TF32:
        return precision
    if int(_lib.load().b200sht_mix_uses_tensor_cores(op & 0xFF, B, G, Ci, Co, precision)):
        return precision
    key = (B, G, Ci, Co)
    if key not in _warned_mix_fallback:
        _warned_mix_fallback.add(key)
        warnings.warn(
            f"makani_b200: the tensor-core channel mix needs a per-GPU batch that divides 32 and group slices that are multiples of 4 channels; "
            f"batch {B}, groups {G}, channels {Ci}->{Co} runs the fp32 CUDA-core mix instead (slower; the SHT stages stay on the tensor cores)",
            RuntimeWarning, stacklevel=3)
    return _lib.PREC_FP32


class PackedWeightCache:
    """Dense operators read the weight in the packed layout float [L][G][Ci/G][cop][2]; the re-layout kernel runs once per
    parameter version (i.e. once per optimizer step in training, never in inference).  `enabled=False` forces it every call."""

    def __init__(self):
        self.enabled = True
        self._key = None
        self._ref = None      # weak reference to the parameter the packed copy was made from
        self._packed = None

    def invalidate(self):
        """Forget the packed copy.  Needed after writes that do not bump the version counter (`weight.data.copy_()`, kernels writing through
        `data_ptr()`); `SpectralConv` / `SpectralAttention` call it from `_apply` and `load_state_dict`."""
        self._key = self._ref = self._packed = None

    def get(self, w, op, L, M, G, Ci, Co, precision=0):
        try:
            version = w._version
        except RuntimeError:     # inference-mode tensors have no version counter: never reuse
            version = None
        key = (w.data_ptr(), version, w.device, op, L, G, Ci, Co, precision)
        same = self._ref is not None and self._ref() is w
        if self.enabled and version is not None and same and self._key == key and self._packed is not None:
            return self._packed
        n = int(_lib.load().b200sht_mix_weight_elems(op, L, M, G, Ci, Co))
        packed = torch.empty(n, dtype=torch.float32, device=w.device)
        wc = w.detach().contiguous()
        _lib.call("b200sht_mix_weight_pack", op, _ptr(wc), _ptr(packed), L, G, Ci, Co, precision, _stream(w.device))
        self._key, self._packed = key, packed
        try:
            self._ref = weakref.ref(w)
        except TypeError:
            self._ref = None
        return packed


class _MixPacked(torch.autograd.Function):
    """y[l,m,b,o] = sum_i x[l,m,b,i] * w[...] on packed spectra (contractions.py:19-151)."""

    @staticmethod
    def forward(ctx, spec, weight, cbias, op, L, M, B, G, Ci, Co, precision, cache):
        dev = spec.device
        spec = spec.contiguous()
        if weight.dtype != torch.complex64:
            raise B200ShtError(f"spectral weights must be complex64, got {weight.dtype}")
        base_op = op & 0xFF  # op may carry _lib.DENSE_FLAG (l/m-sharded spectra of the distributed path)
        if base_op in _DENSE_OPS:
            wdev = (cache if cache is not None else PackedWeightCache()).get(weight, base_op, L, M, G, Ci, Co, mix_pack_precision(base_op, B, G, Ci, Co, precision))
        else:
            wdev = weight.detach().contiguous()
        y = torch.empty(int(_lib.load().b200sht_spec_elems_lm(L, M, B, Co)), dtype=torch.float32, device=dev)
        cb = cbias.detach().reshape(-1).contiguous() if cbias is not None else None
        _lib.call("b200sht_mix_forward", L, M, op, _ptr(spec), _ptr(wdev), _ptr(cb), _ptr(y), B, G, Ci, Co, precision, _stream(dev))
        ctx.save_for_backward(spec, wdev)
        ctx.meta = (op, L, M, B, G, Ci, Co, precision, tuple(weight.shape), tuple(cbias.shape) if cbias is not None else None)
        return y

    @staticmethod
    def backward(ctx, gy):
        spec, wdev = ctx.saved_tensors
        op, L, M, B, G, Ci, Co, precision, wshape, cbshape = ctx.meta
        gy = gy.contiguous()
        dev = gy.device
        lib = _lib.load()
        need_x, need_w, need_cb = ctx.needs_input_grad[0], ctx.needs_input_grad[1], ctx.needs_input_grad[2] and cbshape is not None
        gx = torch.empty(int(lib.b200sht_spec_elems_lm(L, M, B, Ci)), dtype=torch.float32, device=dev) if need_x else None
        gw_dev = None
        base_op = op & 0xFF
        if need_w:
            if base_op in _DENSE_OPS:
                gw_dev = torch.empty(int(lib.b200sht_mix_weight_elems(base_op, L, M, G, Ci, Co)), dtype=torch.float32, device=dev)
            else:
                gw_dev = torch.empty(wshape, dtype=torch.complex64, device=dev)
        gcb = torch.empty(Co, dtype=torch.complex64, device=dev) if need_cb else None
        _lib.call("b200sht_mix_backward", L, M, op, _ptr(spec), _ptr(wdev), _ptr(gy), _ptr(gx), _ptr(gw_dev), _ptr(gcb), B, G, Ci, Co, precision,
                  _stream(dev))
        gw = None
        if need_w:
            if base_op in _DENSE_OPS:
                gw = torch.empty(wshape, dtype=torch.complex64, device=dev)
                _lib.call("b200sht_mix_weight_unpack", base_op, _ptr(gw_dev), _ptr(gw), L, G, Ci, Co, _stream(dev))
            else:
                gw = gw_dev
        if gcb is not None:
            gcb = gcb.reshape(cbshape)
        return gx, gw, gcb, None, None, None, None, None, None, None, None, None


class _SpectralConvOneCall(torch.autograd.Function):
    """SpectralConv forward / backward through b200sht_spectral_conv_forward / _backward (include/b200sht.h)."""

    @staticmethod
    def forward(ctx, x, weight, bias, mod):
        from .sht import _dtype_code
        lib = _lib.load()
        dev = x.device
        B = x.shape[0]
        pf, pi = mod.forward_transform.plan(dev), mod.inverse_transform.plan(dev)
        prec = resolve_precision(mod.precision)
        op = mod._op & 0xFF
        if weight.dtype != torch.complex64:
            raise B200ShtError(f"spectral weights must be complex64, got {weight.dtype}")
        desc = _lib.ConvDesc(B, mod.in_channels, mod.out_channels, mod.num_groups, op, _dtype_code(x.dtype), prec)
        dptr = ctypes.c_void_p(ctypes.addressof(desc))
        wsb = int(lib.b200sht_spectral_conv_workspace_bytes(pf.handle, pi.handle, dptr))
        if wsb < 0:
            _lib.check(-1, "b200sht_spectral_conv_workspace_bytes")
        ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
        L, M = mod.modes_lat_local, mod.modes_lon_local
        if op in _DENSE_OPS:
            wdev = mod._wcache.get(weight, op, L, M, mod.num_groups, mod.in_channels, mod.out_channels,
                                   mix_pack_precision(op, B, mod.num_groups, mod.in_channels, mod.out_channels, prec))
        else:
            wdev = weight.detach().contiguous()
        spec_saved = torch.empty(pf.spec_elems(B, mod.in_channels), dtype=torch.float32, device=dev)
        y = torch.empty((B, mod.out_channels, pi.nlat, pi.nlon), dtype=x.dtype, device=dev)
        res = torch.empty((B, mod.in_channels, pi.nlat, pi.nlon), dtype=x.dtype, device=dev) if mod.scale_residual else None
        b32 = bias.detach().reshape(-1).to(torch.float32).contiguous() if bias is not None else None
        _lib.call("b200sht_spectral_conv_forward", pf.handle, pi.handle, dptr, _ptr(x), _ptr(wdev), _ptr(b32), _ptr(y), _ptr(res), _ptr(spec_saved),
                  _ptr(ws), _stream(dev))
        ctx.save_for_backward(spec_saved, wdev)
        ctx.meta = (pf, pi, (B, mod.in_channels, mod.out_channels, mod.num_groups, op, _dtype_code(x.dtype), prec), tuple(x.shape), x.dtype,
                    tuple(weight.shape), None if bias is None else (tuple(bias.shape), bias.dtype), L, M, wsb)
        ctx.wgrad_event = getattr(mod, "wgrad_ready_event", None)
        return (y, res) if res is not None else y

    @staticmethod
    def backward(ctx, gy, gres=None):
        spec_saved, wdev = ctx.saved_tensors
        pf, pi, d, xshape, xdtype, wshape, binfo, L, M, wsb = ctx.meta
        B, Ci, Co, G, op, dt, prec = d
        lib = _lib.load()
        dev = gy.device
        gy = gy.contiguous().to(xdtype)
        gres = gres.contiguous().to(xdtype) if gres is not None else None
        desc = _lib.ConvDesc(*d)
        dptr = ctypes.c_void_p(ctypes.addressof(desc))
        ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
        need_x, need_w, need_b = ctx.needs_input_grad[0], ctx.needs_input_grad[1], (binfo is not None and ctx.needs_input_grad[2])
        gx = torch.empty(xshape, dtype=xdtype, device=dev) if need_x else None
        gw_dev = None
        if need_w:
            if op in _DENSE_OPS:
                gw_dev = torch.empty(int(lib.b200sht_mix_weight_elems(op, L, M, G, Ci, Co)), dtype=torch.float32, device=dev)
            else:
                gw_dev = torch.empty(wshape, dtype=torch.complex64, device=dev)
        gb = torch.empty(Co, dtype=torch.float32, device=dev) if need_b else None
        # the weight gradient is re-laid-out and its event recorded inside the call, before the input-gradient stages (b200sht.h)
        gw = None
        if need_w:
            gw = torch.empty(wshape, dtype=torch.complex64, device=dev) if op in _DENSE_OPS else gw_dev
        ev = ctx.wgrad_event
        if ev is not None and not ev.cuda_event:
            # torch creates the CUDA event at its first record: without a handle the library would see no event, skip the overlapped
            # schedule, and a stream waiting on the event would not wait for the gradient at all
            ev.record(torch.cuda.current_stream(dev))
        _lib.call("b200sht_spectral_conv_backward_ex", pf.handle, pi.handle, dptr, _ptr(gy), _ptr(gres), _ptr(spec_saved), _ptr(wdev), _ptr(gx), _ptr(gw_dev),
                  _ptr(gb), _ptr(ws), _ptr(gw) if (need_w and op in _DENSE_OPS) else _VP(0), _VP(ev.cuda_event) if ev is not None else _VP(0), _stream(dev))
        gbias = gb.reshape(binfo[0]).to(binfo[1]) if need_b else None
        return gx, gw, gbias, None


def mix_packed(spec, weight, op, L, M, B, G, Ci, Co, precision="auto", cbias=None, cache=None):
    return _MixPacked.apply(spec, weight, cbias, op, L, M, B, G, Ci, Co, resolve_precision(precision), cache)


def _check_transforms(fwd, inv):
    if not (hasattr(fwd, "forward_packed") and hasattr(inv, "forward_packed")):
        raise TypeError(
            "makani_b200.SpectralConv needs makani_b200 transforms (RealSHT/InverseRealSHT or their Distributed* variants); "
            f"got {type(fwd).__name__} / {type(inv).__name__}"
        )


class SpectralConv(nn.Module):
    """Spectral convolution y = iSHT(W . SHT(x)) (+bias); see the reference docstring at spectral_convolution.py:37-114."""

    def __init__(self, forward_transform, inverse_transform, in_channels, out_channels, num_groups=1, operator_type="dhconv", separable=False,
                 bias=False, gain=1.0, precision="auto"):
        super().__init__()
        if in_channels % num_groups != 0:
            raise ValueError(f"in_channels ({in_channels}) must be divisible by num_groups ({num_groups})")
        if out_channels % num_groups != 0:
            raise ValueError(f"out_channels ({out_channels}) must be divisible by num_groups ({num_groups})")
        _check_transforms(forward_transform, inverse_transform)

        self.forward_transform = forward_transform
        self.inverse_transform = inverse_transform
        self.in_channels, self.out_channels, self.num_groups = in_channels, out_channels, num_groups
        self.modes_lat = self.inverse_transform.lmax
        self.modes_lon = self.inverse_transform.mmax
        self.scale_residual = (self.forward_transform.nlat != self.inverse_transform.nlat) or (self.forward_transform.nlon != self.inverse_transform.nlon)
        if hasattr(self.forward_transform, "grid"):
            self.scale_residual = self.scale_residual or (self.forward_transform.grid != self.inverse_transform.grid)
        self.operator_type, self.separable, self.precision = operator_type, separable, precision

        if self.forward_transform.lmax != self.modes_lat:
            raise ValueError(f"inverse transform lmax ({self.inverse_transform.lmax}) must match modes_lat ({self.forward_transform.lmax})")
        if self.forward_transform.mmax != self.modes_lon:
            raise ValueError(f"inverse transform mmax ({self.inverse_transform.mmax}) must match modes_lon ({self.forward_transform.mmax})")
        if operator_type not in ("diagonal", "dhconv"):
            raise ValueError(f"Unsupported operator type f{operator_type}")
        if separable and in_channels != out_channels:
            raise ValueError("separable spectral convolution requires out_channels == in_channels")

        weight_shape = [num_groups, in_channels // num_groups]
        if not separable:
            weight_shape += [out_channels // num_groups]

        # local (possibly sharded) mode counts: distributed transforms publish their shard via l_local / m_local
        self.modes_lat_local = getattr(self.inverse_transform, "lmax_local", self.modes_lat)
        self.modes_lon_local = getattr(self.inverse_transform, "mmax_local", self.modes_lon)
        self.nlat_local = getattr(self.inverse_transform, "nlat_local", self.inverse_transform.nlat)
        self.nlon_local = getattr(self.inverse_transform, "nlon_local", self.inverse_transform.nlon)

        if operator_type == "diagonal":
            weight_shape += [self.modes_lat_local, self.modes_lon_local]
        else:
            weight_shape += [self.modes_lat_local]

        # initialisation as spectral_convolution.py:189-193 (l = 0 of the local shard scaled by sqrt 2)
        scale = math.sqrt(gain / (in_channels // num_groups)) * torch.ones(self.modes_lat_local, dtype=torch.complex64)
        scale[0] *= math.sqrt(2.0)
        if operator_type == "diagonal":
            init = scale.reshape(-1, 1) * torch.randn(*weight_shape, dtype=torch.complex64)
        else:
            init = scale * torch.randn(*weight_shape, dtype=torch.complex64)
        self.weight = nn.Parameter(init)
        if operator_type == "dhconv":
            self.weight.is_shared_mp = ["matmul", "w"]
            self.weight.sharded_dims_mp = [None for _ in weight_shape]
            self.weight.sharded_dims_mp[-1] = "h"
        else:
            self.weight.is_shared_mp = ["matmul"]
            self.weight.sharded_dims_mp = [None for _ in weight_shape]
            self.weight.sharded_dims_mp[-1] = "w"
            self.weight.sharded_dims_mp[-2] = "h"

        if bias == True:  # noqa: E712  (same test as the reference)
            self.bias = nn.Parameter(torch.zeros(1, self.out_channels, 1, 1))
            self.bias.is_shared_mp = ["model"]
            self.bias.sharded_dims_mp = [None, None, None, None]

        self._op = _op_code(operator_type, separable)
        if getattr(self.inverse_transform, "packed_dense", False):
            self._op |= _lib.DENSE_FLAG
        self._wcache = PackedWeightCache()
        self.one_call = True   # False: one autograd node per stage (same kernels; used by the distributed transforms)

    def invalidate_weight_cache(self):
        """after writes to `weight` that bypass the version counter (`weight.data.copy_`, custom kernels)"""
        self._wcache.invalidate()

    def _apply(self, fn, *args, **kwargs):           # .to() / .cuda() / .float(): the parameter storage changes
        self._wcache.invalidate()
        return super()._apply(fn, *args, **kwargs)

    def _load_from_state_dict(self, *args, **kwargs):
        self._wcache.invalidate()
        return super()._load_from_state_dict(*args, **kwargs)

    def forward(self, x):
        dtype = x.dtype
        residual = x
        xin = x if dtype in (torch.float32, torch.bfloat16) else x.to(torch.float32)
        out_dtype = xin.dtype
        B = xin.shape[0]
        if self.one_call and isinstance(self.forward_transform, RealSHT) and isinstance(self.inverse_transform, InverseRealSHT):
            # whole block through the two C-ABI entry points b200sht_spectral_conv_forward / _backward (2 host calls per step)
            bias = self.bias if hasattr(self, "bias") else None
            out = _SpectralConvOneCall.apply(xin.contiguous(), self.weight, bias, self)
            if self.scale_residual:
                return out[0].to(dtype), out[1].to(dtype)
            return out.to(dtype), residual
        # transforms run in fp32/TF32 regardless of autocast, as the reference disables autocast around them (:237-241)
        xs = self.forward_transform.forward_packed(xin)
        if self.scale_residual:
            residual = self.inverse_transform.forward_packed(xs, B, self.in_channels, out_dtype).to(dtype)
        ys = mix_packed(xs, self.weight, self._op, self.modes_lat_local, self.modes_lon_local, B, self.num_groups, self.in_channels,
                        self.out_channels, self.precision, cache=self._wcache)
        bias = self.bias if hasattr(self, "bias") else None
        y = self.inverse_transform.forward_packed(ys, B, self.out_channels, out_dtype, bias=bias).to(dtype)
        return y, residual


# ----------------------------------------------------------------------------------------------------------------
# ComplexReLU / SpectralAttention
# ----------------------------------------------------------------------------------------------------------------
_RELU_MODES = {"real": 0, "cartesian": 1, "modulus": 2, "halfplane": 3}


class _ComplexReLUPacked(torch.autograd.Function):
    @staticmethod
    def forward(ctx, spec, bias, mode, slope, L, M, B, C):
        spec = spec.contiguous()
        y = torch.empty_like(spec)
        b = bias.detach().reshape(-1).to(torch.float32).contiguous() if bias is not None else None
        if b is not None and b.numel() == 1:
            b = b.expand(C).contiguous()
        _lib.call("b200sht_complex_relu_forward", L, M, mode, _ptr(spec), _ptr(b), float(slope), _ptr(y), B, C, _stream(spec.device))
        ctx.save_for_backward(spec, b)
        ctx.meta = (mode, slope, L, M, B, C, tuple(bias.shape) if bias is not None else None)
        return y

    @staticmethod
    def backward(ctx, gy):
        spec, b = ctx.saved_tensors
        mode, slope, L, M, B, C, bshape = ctx.meta
        gy = gy.contiguous()
        gx = torch.empty_like(spec)
        need_b = bshape is not None and ctx.needs_input_grad[1] and (mode & 0xFF) == 2
        gb = torch.empty(C, dtype=torch.float32, device=gy.device) if need_b else None
        _lib.call("b200sht_complex_relu_backward", L, M, mode, _ptr(spec), _ptr(b), float(slope), _ptr(gy), _ptr(gx), _ptr(gb), B, C,
                  _stream(gy.device))
        gbias = None
        if bshape is not None and ctx.needs_input_grad[1]:
            if gb is None:
                gbias = torch.zeros(bshape, dtype=torch.float32, device=gy.device)
            else:
                n = 1
                for s in bshape:
                    n *= s
                gbias = gb.sum().reshape(bshape) if n == 1 else gb.reshape(bshape)
        return gx, gbias, None, None, None, None, None, None


class ComplexReLU(nn.Module):
    """Complex rectifier (modes real / cartesian / modulus / halfplane), mirror of activations.py:20-127."""

    def __init__(self, negative_slope=0.0, mode="real", bias_shape=None, scale=1.0):
        super().__init__()
        self.mode = mode
        if self.mode in ["modulus", "halfplane"]:
            if bias_shape is not None:
                self.bias = nn.Parameter(scale * torch.ones(bias_shape, dtype=torch.float32))
            else:
                self.bias = nn.Parameter(scale * torch.ones((1), dtype=torch.float32))
        else:
            self.bias = 0
        self.negative_slope = negative_slope

    def forward_packed(self, spec, L, M, B, C, dense=False):
        if self.mode not in _RELU_MODES:
            raise NotImplementedError
        bias = self.bias if isinstance(self.bias, torch.Tensor) else None
        mode = _RELU_MODES[self.mode] | (_lib.DENSE_FLAG if dense else 0)
        return _ComplexReLUPacked.apply(spec, bias, mode, self.negative_slope, L, M, B, C)

    def forward(self, z):
        if self.mode not in _RELU_MODES:
            raise NotImplementedError
        z4 = z if z.dim() == 4 else z.reshape(1, -1, *z.shape[-2:])
        B, C, L, M = z4.shape
        out = _SpecUnpack.apply(self.forward_packed(_SpecPack.apply(z4.to(torch.complex64)), L, M, B, C), L, M, B, C)
        return out.reshape(z.shape)


class SpectralAttention(nn.Module):
    """Complex MLP in spectral space.  The reference's forward raises at HEAD (SURVEY.md F3); this implements the intended
    semantics: per layer h = ComplexReLU(einsum("bixy,io->boxy" | "bixy,xio->boxy", h, w) (+b)), then the output mix."""

    def __init__(self, forward_transform, inverse_transform, in_channels, out_channels, operator_type="diagonal", hidden_size_factor=2,
                 complex_activation="real", bias=False, spectral_layers=1, drop_rate=0.0, gain=1.0, precision="auto"):
        super().__init__()
        _check_transforms(forward_transform, inverse_transform)
        self.in_channels, self.out_channels = in_channels, out_channels
        self.operator_type, self.spectral_layers, self.precision = operator_type, spectral_layers, precision
        self.modes_lat, self.modes_lon = forward_transform.lmax, forward_transform.mmax
        self.forward_transform, self.inverse_transform = forward_transform, inverse_transform
        self.scale_residual = ((forward_transform.nlat != inverse_transform.nlat) or (forward_transform.nlon != inverse_transform.nlon)
                               or (forward_transform.grid != inverse_transform.grid))
        if inverse_transform.lmax != self.modes_lat:
            raise ValueError(f"inverse transform lmax ({inverse_transform.lmax}) must match modes_lat ({self.modes_lat})")
        if inverse_transform.mmax != self.modes_lon:
            raise ValueError(f"inverse transform mmax ({inverse_transform.mmax}) must match modes_lon ({self.modes_lon})")
        hidden = int(hidden_size_factor * in_channels)
        self.hidden_size = hidden
        if operator_type == "diagonal":
            lead = []
            self._op = _lib.OP_SHARED
        elif operator_type == "l-dependant":
            lead = [self.modes_lat]
            self._op = _lib.OP_LDEP
        else:
            raise ValueError("Unknown operator type")
        scale = math.sqrt(2.0 / float(in_channels))
        w = [scale * torch.randn(*lead, in_channels, hidden, dtype=torch.complex64)]
        for _ in range(1, spectral_layers):
            scale = math.sqrt(2.0 / float(hidden))
            w.append(scale * torch.randn(*lead, hidden, hidden, dtype=torch.complex64))
        self.w = nn.ParameterList(w)
        scale_b = scale if operator_type == "l-dependant" else math.sqrt(gain / float(in_channels))
        if operator_type == "diagonal":
            scale = math.sqrt(gain / float(in_channels))
            self.wout = nn.Parameter(scale * torch.randn(hidden, out_channels, dtype=torch.complex64))
            if bias:
                self.b = nn.ParameterList([scale * torch.randn(hidden, 1, 1, dtype=torch.complex64) for _ in range(spectral_layers)])
        else:
            if bias:
                self.b = nn.ParameterList([scale_b * torch.randn(hidden, 1, 1, dtype=torch.complex64) for _ in range(spectral_layers)])
            scale = math.sqrt(gain / float(in_channels))
            self.wout = nn.Parameter(scale * torch.randn(self.modes_lat, hidden, out_channels, dtype=torch.complex64))
        self.activations = nn.ModuleList([ComplexReLU(mode=complex_activation, bias_shape=(hidden, 1, 1), scale=scale) for _ in range(spectral_layers)])
        # the reference builds nn.Dropout here (spectral_convolution.py:432); dropout on packed spectra is not implemented, so the
        # constructor accepts drop_rate (configs load unchanged) and forward() raises when it would actually drop (training, p > 0)
        self.drop_rate = float(drop_rate)
        self.drop = nn.Dropout(drop_rate) if drop_rate > 0.0 else nn.Identity()
        self._caches = [PackedWeightCache() for _ in range(spectral_layers + 1)]
        # l / m-sharded spectra (Distributed* transforms of the h x w path): the packed buffers hold the LOCAL modes, every (l, m) stored
        self.modes_lat_local = getattr(inverse_transform, "lmax_local", self.modes_lat)
        self.modes_lon_local = getattr(inverse_transform, "mmax_local", self.modes_lon)
        self._dense = _lib.DENSE_FLAG if getattr(inverse_transform, "packed_dense", False) else 0
        if operator_type == "l-dependant" and self.modes_lat_local != self.modes_lat:
            raise ValueError("SpectralAttention(operator_type='l-dependant') with an l-sharded transform (h_parallel_size > 1) is not supported: "
                             "its weights are indexed by the global degree")

    def invalidate_weight_cache(self):
        for c in self._caches:
            c.invalidate()

    def _apply(self, fn, *args, **kwargs):
        self.invalidate_weight_cache()
        return super()._apply(fn, *args, **kwargs)

    def _load_from_state_dict(self, *args, **kwargs):
        self.invalidate_weight_cache()
        return super()._load_from_state_dict(*args, **kwargs)

    def _mlp_packed(self, h, B):
        if self.training and self.drop_rate > 0.0:
            raise NotImplementedError("SpectralAttention: dropout on complex spectra (drop_rate > 0 in training) is not implemented")
        L, M = self.modes_lat_local, self.modes_lon_local
        op = self._op | self._dense
        cin = self.in_channels
        for i in range(self.spectral_layers):
            cb = self.b[i] if hasattr(self, "b") else None
            h = mix_packed(h, self.w[i], op, L, M, B, 1, cin, self.hidden_size, self.precision, cbias=cb, cache=self._caches[i])
            h = self.activations[i].forward_packed(h, L, M, B, self.hidden_size, dense=bool(self._dense))
            cin = self.hidden_size
        return mix_packed(h, self.wout, op, L, M, B, 1, cin, self.out_channels, self.precision, cache=self._caches[-1])

    def forward_mlp(self, x):
        """complex (B, Cin, L, M) -> complex (B, Cout, L, M)."""
        B, C, L, M = x.shape
        out = self._mlp_packed(_SpecPack.apply(x.to(torch.complex64)), B)
        return _SpecUnpack.apply(out, L, M, B, self.out_channels)

    def forward(self, x):
        dtype = x.dtype
        residual = x
        xin = x if dtype in (torch.float32, torch.bfloat16) else x.to(torch.float32)
        B = xin.shape[0]
        xs = self.forward_transform.forward_packed(xin)
        if self.scale_residual:
            residual = self.inverse_transform.forward_packed(xs, B, self.in_channels, xin.dtype).to(dtype)
        ys = self._mlp_packed(xs, B)
        y = self.inverse_transform.forward_packed(ys, B, self.out_channels, xin.dtype).to(dtype)
        return y, residual
