"""SFNO network around the CUDA spherical-harmonic path: the callers of SpectralConv / SpectralAttention (SURVEY rows A8, A9).

Restates, with the same constructor arguments, parameter names, shapes, initialisation scales and model-parallel tags, the reference's
  NeuralOperatorBlock                 makani/models/networks/sfnonet.py:169-408   (filter -> norm0 -> [+inner skip] -> act -> MLP -> norm1 -> drop path -> [+outer skip])
  SphericalFourierNeuralOperatorNet   makani/models/networks/sfnonet.py:411-934   (encoder, position embedding, blocks, decoder, big skip; `_init_spectral_transforms` :765-838)
  MLP / EncoderDecoder                makani/models/common/layers.py:537-760      (1x1-convolution stacks, `fwd` Sequential)
so that a checkpoint of the reference network loads with `load_state_dict(strict=True)` and gives the same outputs (tests/golden/sfno_golden_<case>.npz is
produced by the REFERENCE class here, tests/golden/make_sfno_golden.py).  Single-process (h = w = 1) SHT variant; the makani package itself can also
be run unchanged on these kernels through makani_b200.compat (torch_harmonics shim).

`backend` lets the same network be built on other transform / filter classes (bench.py's CPU reference arm passes the oracle's).
"""
import math
from functools import partial

import torch
import torch.nn as nn
from torch import amp

_ACTS = {"relu": nn.ReLU, "gelu": nn.GELU, "silu": nn.SiLU}


def _tag_spatial(p):
    p.is_shared_mp = ["spatial"]     # pointwise layers hold identical parameters on every spatial rank (layers.py:611-617)
    return p


class Conv1x1(nn.Conv2d):
    """`nn.Conv2d(cin, cout, 1)` with the reference's parameter names / shapes / init (weight [cout, cin, 1, 1], bias [cout]) whose forward is the
    plain GEMM `W [cout, cin] @ x [B, cin, H*W]` on the NCHW tensor itself.  cuDNN runs a bf16 1x1 convolution as an NHWC implicit GEMM between two
    layout conversions of the whole activation (profile of the sfno_sc3_layers8_edim384 step: 66 `nchwToNhwc` / `nhwcToNchw` launches, 11.5 ms of a
    77 ms step); the longitude transforms on either side need NCHW, so the GEMM is done in that layout (cuBLAS, a library GEMM) and the conversions
    disappear.  Same arithmetic (bf16 operands under autocast, fp32 accumulation), same gradients."""

    def is_plain(self, x):
        return self.groups == 1 and x.dim() == 4 and self.kernel_size == (1, 1) and self.padding_mode == "zeros"

    def gemm(self, x):
        """W @ x without the bias (the caller adds it, or fuses it with the activation that follows: `_run_stack`)"""
        B, C, H, W = x.shape
        w = self.weight.view(1, self.out_channels, self.in_channels)
        if w.dtype != x.dtype and x.dtype in (torch.bfloat16, torch.float16):
            w = w.to(x.dtype)            # activations already in the autocast dtype: cast the (small) weight once, before the batch expansion
        # bmm on (B, cout, cin) x (B, cin, H*W): the output is the contiguous NCHW tensor.  (torch.matmul(2-D, 3-D) folds the batch into the rows of the
        # TRANSPOSED problem and hands back a transposed view: the copy that makes it contiguous cost 50 ms per model step when this was first measured.)
        return torch.bmm(w.expand(B, -1, -1), x.reshape(B, C, H * W)).view(B, self.out_channels, H, W)

    def forward(self, x):
        if not self.is_plain(x):
            return super().forward(x)
        y = self.gemm(x)
        if self.bias is not None:
            y = y + self.bias.to(y.dtype).view(1, -1, 1, 1)
        return y


def _run_stack(mods, x):
    """nn.Sequential of 1x1 convolutions, activations and dropouts, with `conv -> (+ bias) -> GELU` as GEMM + one fused bias + GELU kernel
    (makani_b200.norm.bias_gelu) where the pattern and the device allow it; otherwise module by module."""
    from .norm import bias_gelu, fused_pointwise_enabled

    mods = list(mods)
    i = 0
    while i < len(mods):
        m = mods[i]
        nxt = mods[i + 1] if i + 1 < len(mods) else None
        if (isinstance(m, Conv1x1) and isinstance(nxt, nn.GELU) and getattr(nxt, "approximate", "none") == "none" and x.is_cuda and fused_pointwise_enabled()
                and m.is_plain(x)):
            x = bias_gelu(m.gemm(x), m.bias)
            i += 2
        else:
            x = m(x)
            i += 1
    return x


class DropPath(nn.Module):
    """stochastic depth per sample (layers.py:49-90)"""

    def __init__(self, drop_prob=0.0):
        super().__init__()
        self.drop_prob = drop_prob

    def forward(self, x):
        if self.drop_prob == 0.0 or not self.training:
            return x
        keep = 1.0 - self.drop_prob
        mask = x.new_empty((x.shape[0],) + (1,) * (x.ndim - 1)).bernoulli_(keep)
        return x.div(keep) * mask


class EncoderDecoder(nn.Module):
    """`num_layers` x (1x1 conv + activation) and a bias-free output projection; He init, output std sqrt(gain / fan_in)."""

    def __init__(self, num_layers, input_dim, output_dim, hidden_dim, act_layer, gain=1.0, input_format="nchw", groups=1):
        super().__init__()
        if input_format != "nchw":
            raise NotImplementedError(f"Error, input format {input_format} not supported.")
        mods, cur = [], input_dim
        for _ in range(num_layers):
            conv = Conv1x1(cur, hidden_dim, 1, bias=True, groups=groups)
            nn.init.normal_(_tag_spatial(conv.weight), mean=0.0, std=math.sqrt(2.0 / (cur // groups)))
            nn.init.constant_(_tag_spatial(conv.bias), 0.0)
            mods += [conv, act_layer()]
            cur = hidden_dim
        out = Conv1x1(cur, output_dim, 1, bias=False, groups=groups)
        nn.init.normal_(_tag_spatial(out.weight), mean=0.0, std=math.sqrt(gain / (cur // groups)))
        mods.append(out)
        self.fwd = nn.Sequential(*mods)

    def forward(self, x):
        return _run_stack(self.fwd, x)


class MLP(nn.Module):
    """fc1 -> act -> drop -> fc2 -> drop as 1x1 convolutions (state-dict keys fwd.0 / fwd.3, as the reference's)."""

    def __init__(self, in_features, hidden_features=None, out_features=None, act_layer=nn.GELU, output_bias=True, drop_rate=0.0, drop_type="iid",
                 gain=1.0, **kwargs):
        super().__init__()
        out_features = out_features or in_features
        hidden_features = hidden_features or in_features
        fc1 = Conv1x1(in_features, hidden_features, 1, bias=True)
        fc2 = Conv1x1(hidden_features, out_features, 1, bias=output_bias)
        nn.init.normal_(_tag_spatial(fc1.weight), mean=0.0, std=math.sqrt(2.0 / in_features))
        nn.init.constant_(_tag_spatial(fc1.bias), 0.0)
        nn.init.normal_(_tag_spatial(fc2.weight), mean=0.0, std=math.sqrt(gain / hidden_features))
        if fc2.bias is not None:
            nn.init.constant_(_tag_spatial(fc2.bias), 0.0)
        if drop_rate > 0.0:
            if drop_type not in ("iid", "features"):
                raise NotImplementedError(f"Error, drop_type {drop_type} not supported")
            drop = nn.Dropout(drop_rate) if drop_type == "iid" else nn.Dropout2d(drop_rate)
        else:
            drop = nn.Identity()
        self.fwd = nn.Sequential(fc1, act_layer(), drop, fc2, drop)

    def forward(self, x):
        return _run_stack(self.fwd, x)


class _Backend:
    """default classes: the CUDA path of this package"""

    def __init__(self, precision="auto"):
        import makani_b200 as mb

        self.RealSHT = partial(mb.RealSHT, precision=precision)
        self.InverseRealSHT = partial(mb.InverseRealSHT, precision=precision)
        self.SpectralConv = partial(mb.SpectralConv, precision=precision)
        self.SpectralAttention = partial(mb.SpectralAttention, precision=precision)


class SpectralFilterLayer(nn.Module):
    """linear (SpectralConv) or non-linear (SpectralAttention) filter; parameters live under `.filter` (sfnonet.py:52-167)"""

    def __init__(self, forward_transform, inverse_transform, embed_dim, filter_type="linear", operator_type="diagonal", hidden_size_factor=1,
                 rank=1.0, separable=False, complex_activation="real", spectral_layers=1, bias=False, drop_rate=0.0, gain=1.0, backend=None):
        super().__init__()
        backend = backend or _Backend()
        if filter_type == "non-linear":
            self.filter = backend.SpectralAttention(forward_transform, inverse_transform, embed_dim, embed_dim, operator_type=operator_type,
                                                    hidden_size_factor=hidden_size_factor, complex_activation=complex_activation,
                                                    spectral_layers=spectral_layers, drop_rate=drop_rate, bias=bias, gain=gain)
        elif filter_type == "linear":
            self.filter = backend.SpectralConv(forward_transform, inverse_transform, embed_dim, embed_dim, operator_type=operator_type,
                                               separable=separable, bias=bias, gain=gain)
        else:
            raise NotImplementedError

    def forward(self, x):
        return self.filter(x)


class NeuralOperatorBlock(nn.Module):
    def __init__(self, forward_transform, inverse_transform, embed_dim, filter_type="linear", operator_type="diagonal", mlp_ratio=2.0, mlp_drop_rate=0.0,
                 path_drop_rate=0.0, act_layer=nn.GELU, norm_layer=(nn.Identity, nn.Identity), rank=1.0, separable=False, inner_skip="linear",
                 outer_skip=None, use_mlp=False, comm_feature_name="matmul", complex_activation="real", spectral_layers=1, bias=False,
                 final_activation=False, checkpointing_level=0, backend=None):
        super().__init__()
        self.input_shape_loc = (forward_transform.nlat, forward_transform.nlon)
        self.output_shape_loc = (inverse_transform.nlat, inverse_transform.nlon)
        self.norm0 = norm_layer[0]()
        gain = 1.0 if act_layer == nn.Identity else 2.0
        gain = self._make_skip("inner_skip", inner_skip, embed_dim, gain)
        self.filter = SpectralFilterLayer(forward_transform, inverse_transform, embed_dim, filter_type, operator_type, hidden_size_factor=mlp_ratio,
                                          rank=rank, separable=separable, complex_activation=complex_activation, spectral_layers=spectral_layers,
                                          bias=bias, drop_rate=path_drop_rate, gain=gain, backend=backend)
        self.act_layer0 = act_layer()
        self.norm1 = norm_layer[1]()
        gain = 2.0 if (final_activation and act_layer != nn.Identity) else 1.0
        gain = self._make_skip("outer_skip", outer_skip, embed_dim, gain)
        if use_mlp:
            self.mlp = MLP(in_features=embed_dim, hidden_features=int(embed_dim * mlp_ratio), act_layer=act_layer, drop_rate=mlp_drop_rate,
                           drop_type="features", gain=gain)
        self.drop_path = DropPath(path_drop_rate) if path_drop_rate > 0.0 else nn.Identity()
        if final_activation:
            self.act_layer1 = act_layer()

    def _make_skip(self, name, kind, embed_dim, gain):
        """'linear': 1x1 conv initialised with half the variance budget; 'identity'; 'none' (no attribute at all, as the reference)."""
        if kind == "linear":
            conv = Conv1x1(embed_dim, embed_dim, 1, 1, bias=False)
            gain /= 2.0
            nn.init.normal_(conv.weight, std=math.sqrt(gain / embed_dim))
            setattr(self, name, conv)
        elif kind == "identity":
            setattr(self, name, nn.Identity())
            gain /= 2.0
        elif kind != "none":
            raise ValueError(f"Unknown skip connection type {kind}")
        return gain

    def forward(self, x):
        from .norm import InstanceNorm2d as FusedInstanceNorm2d

        x, residual = self.filter(x)
        if (isinstance(self.norm0, FusedInstanceNorm2d) and not hasattr(self, "inner_skip") and isinstance(self.act_layer0, nn.GELU)
                and getattr(self.act_layer0, "approximate", "none") == "none"):
            x = self.norm0(x, gelu=True)     # norm0 -> GELU in one pass (sfnonet.py:387-392 with inner_skip "none")
        else:
            x = self.norm0(x)
            if hasattr(self, "inner_skip"):
                x = x + self.inner_skip(residual)
            x = self.act_layer0(x)
        if hasattr(self, "mlp"):
            x = self.mlp(x)
        x = self.drop_path(self.norm1(x))
        if hasattr(self, "outer_skip"):
            x = x + self.outer_skip(residual)
        if hasattr(self, "act_layer1"):
            x = self.act_layer1(x)
        return x


class SphericalFourierNeuralOperatorNet(nn.Module):
    def __init__(self, spectral_transform="sht", model_grid_type="equiangular", sht_grid_type="legendre-gauss", filter_type="linear", operator_type="dhconv",
                 inp_shape=(721, 1440), out_shape=(721, 1440), scale_factor=8, inp_chans=2, out_chans=2, embed_dim=32, num_layers=4, use_mlp=True,
                 mlp_ratio=2.0, encoder_ratio=1, decoder_ratio=1, activation_function="gelu", encoder_layers=1, pos_embed="none", pos_drop_rate=0.0,
                 path_drop_rate=0.0, mlp_drop_rate=0.0, normalization_layer="instance_norm", max_modes=None, hard_thresholding_fraction=1.0, big_skip=True,
                 rank=1.0, separable=False, complex_activation="real", spectral_layers=3, bias=False, checkpointing_level=0, precision="auto", backend=None,
                 **kwargs):
        super().__init__()
        if spectral_transform != "sht":
            raise ValueError("Unknown spectral transform" if spectral_transform != "fft" else "makani_b200.sfno implements the SHT variant only")
        if activation_function not in _ACTS:
            raise ValueError(f"Unknown activation function {activation_function}")
        act = _ACTS[activation_function]
        backend = backend or _Backend(precision)
        self.inp_shape, self.out_shape = tuple(inp_shape), tuple(out_shape)
        self.inp_chans, self.out_chans, self.embed_dim = inp_chans, out_chans, embed_dim
        self.big_skip, self.checkpointing_level = big_skip, checkpointing_level
        self.h, self.w = int(self.inp_shape[0] // scale_factor), int(self.inp_shape[1] // scale_factor)
        self._init_spectral_transforms(backend, model_grid_type, sht_grid_type, hard_thresholding_fraction, max_modes)

        self.encoder = EncoderDecoder(num_layers=encoder_layers, input_dim=inp_chans, output_dim=embed_dim, hidden_dim=int(encoder_ratio * embed_dim),
                                      act_layer=act, input_format="nchw")
        self.pos_drop = nn.Dropout(p=pos_drop_rate) if pos_drop_rate > 0.0 else nn.Identity()
        dpr = [v.item() for v in torch.linspace(0, path_drop_rate, num_layers)]

        if normalization_layer == "instance_norm":
            from .norm import InstanceNorm2d as FusedInstanceNorm2d   # nn.InstanceNorm2d subclass: same parameters / state dict, CUDA kernels of csrc/norm.cu

            norm = partial(FusedInstanceNorm2d, num_features=embed_dim, eps=1e-6, affine=True, track_running_stats=False)
        elif normalization_layer == "none":
            norm = nn.Identity
        else:
            raise NotImplementedError(f"Error, normalization {normalization_layer} not implemented.")

        self.blocks = nn.ModuleList()
        for i in range(num_layers):
            fwd = self.trans_down if i == 0 else self.trans
            inv = self.itrans_up if i == num_layers - 1 else self.itrans
            self.blocks.append(NeuralOperatorBlock(fwd, inv, embed_dim, filter_type=filter_type, operator_type=operator_type, mlp_ratio=mlp_ratio,
                                                   mlp_drop_rate=mlp_drop_rate, path_drop_rate=dpr[i], act_layer=act, norm_layer=(norm, norm),
                                                   inner_skip="none", outer_skip="linear", use_mlp=use_mlp, rank=rank, separable=separable,
                                                   complex_activation=complex_activation, spectral_layers=spectral_layers, bias=bias,
                                                   checkpointing_level=checkpointing_level, backend=backend))

        self.decoder = EncoderDecoder(num_layers=encoder_layers, input_dim=embed_dim, output_dim=out_chans, hidden_dim=int(decoder_ratio * embed_dim),
                                      act_layer=act, gain=0.5 if big_skip else 1.0, input_format="nchw")
        if big_skip:
            self.residual_transform = Conv1x1(inp_chans, out_chans, 1, bias=False)
            self.residual_transform.weight.is_shared_mp = ["spatial"]
            self.residual_transform.weight.sharded_dims_mp = [None, None, None, None]
            nn.init.normal_(self.residual_transform.weight, mean=0.0, std=math.sqrt(0.5 / inp_chans))

        if pos_embed == "direct":
            self.pos_embed = nn.Parameter(torch.zeros(1, embed_dim, *self.inp_shape_loc))
            self.pos_embed.is_shared_mp, self.pos_embed.sharded_dims_mp, self.pos_embed.type = [], [None, None, "h", "w"], "direct"
            with torch.no_grad():
                nn.init.trunc_normal_(self.pos_embed, std=0.02)
        elif pos_embed == "frequency":
            L, M = self.itrans_up.lmax, self.itrans_up.mmax
            rc = nn.Parameter(torch.tril(torch.randn(1, embed_dim, L, M), diagonal=0))
            cc = nn.Parameter(torch.tril(torch.randn(1, embed_dim, L, M - 1), diagonal=-1))
            with torch.no_grad():
                nn.init.trunc_normal_(rc, std=0.02)
                nn.init.trunc_normal_(cc, std=0.02)
            self.pos_embed = nn.ParameterList([rc, cc])
            self.pos_embed.type, self.pos_embed.is_shared_mp, self.pos_embed.sharded_dims_mp = "frequency", [], [None, None, "h", "w"]
        elif pos_embed not in ("none", "None", None):
            raise ValueError("Unknown position embedding type")

    def _init_spectral_transforms(self, backend, model_grid_type, sht_grid_type, hard_thresholding_fraction, max_modes):
        """four transforms: outer grid in (trans_down) / out (itrans_up), inner (h, w) grid both ways; modes = int(h * frac), int((w // 2 + 1) * frac)"""
        if max_modes is not None:
            modes_lat, modes_lon = max_modes
        else:
            modes_lat = int(self.h * hard_thresholding_fraction)
            modes_lon = int((self.w // 2 + 1) * hard_thresholding_fraction)
        self.trans_down = backend.RealSHT(*self.inp_shape, lmax=modes_lat, mmax=modes_lon, grid=model_grid_type).float()
        self.itrans_up = backend.InverseRealSHT(*self.out_shape, lmax=modes_lat, mmax=modes_lon, grid=model_grid_type).float()
        self.trans = backend.RealSHT(self.h, self.w, lmax=modes_lat, mmax=modes_lon, grid=sht_grid_type).float()
        self.itrans = backend.InverseRealSHT(self.h, self.w, lmax=modes_lat, mmax=modes_lon, grid=sht_grid_type).float()
        self.inp_shape_loc = (self.trans_down.nlat, self.trans_down.nlon)
        self.out_shape_loc = (self.itrans_up.nlat, self.itrans_up.nlon)
        self.h_loc, self.w_loc = self.itrans.nlat, self.itrans.nlon

    def no_weight_decay(self):
        return {"pos_embed", "cls_token"}

    def _run(self, fn, x, level):
        if self.checkpointing_level >= level:
            from torch.utils.checkpoint import checkpoint

            return checkpoint(fn, x, use_reentrant=False)
        return fn(x)

    def forward(self, x):
        if self.big_skip:
            residual = x
            if self.out_shape != self.inp_shape:     # resample the skip through the outer transforms, in fp32
                with amp.autocast(device_type=x.device.type, enabled=False):
                    residual = self.itrans_up(self.trans_down(x.to(torch.float32)).contiguous()).to(dtype=x.dtype)
        x = self._run(self.encoder, x, 1)
        if hasattr(self, "pos_embed"):
            pe = self.pos_embed
            if pe.type == "frequency":
                coeffs = torch.stack([pe[0], nn.functional.pad(pe[1], (1, 0), "constant", 0)], dim=-1)
                with amp.autocast(device_type=x.device.type, enabled=False):
                    pe = self.itrans_up(torch.view_as_complex(coeffs))
            x = x + pe.to(dtype=x.dtype)
        x = self.pos_drop(x)
        for blk in self.blocks:
            x = self._run(blk, x, 3)
        x = self._run(self.decoder, x, 1)
        if self.big_skip:
            x = x + self.residual_transform(residual)
        return x
