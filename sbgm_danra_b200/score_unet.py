"""Drop-in mirror of the reference's `sbgm/score_unet.py` import surface, executing on sm_100a kernels.

Same class names, constructor signatures, forward signatures, error behaviour and state-dict keys
(the checkpoint ABI, SURVEY.md section 5) as the reference; the modules below are *parameter
containers* -- their `forward` hands the tensors to `engine.py`, which sequences the CUDA
kernels of `include/sbgm_b200.h`.  Nothing here computes with torch operators on the hot path and
nothing falls back to the CPU.

Reference locations: SinusoidalEmbedding score_unet.py:24-45, ImageSelfAttention :112-148,
Encoder :151-397, DecoderBlock :409-627, Decoder :662-789, ScoreNet :792-879,
marginal_prob_std :881-897, diffusion_coeff :916-930, loss_fn :936-985.
"""
from __future__ import annotations

import functools
import logging
import os
from typing import Iterable, List, Optional, Tuple

import torch
import torch.nn as nn

from . import engine as _eng
from ._lib import call

logger = logging.getLogger(__name__)

DEFAULT_PRECISION = os.environ.get("SBGM_B200_PRECISION", "bf16x3")


def _default_device(device=None) -> torch.device:
    return torch.device(device) if device is not None else torch.device("cuda" if torch.cuda.is_available() else "cpu")


def _act_name(activation) -> str:
    if isinstance(activation, str):
        return activation.lower()
    for cls, name in ((nn.SiLU, "silu"), (nn.GELU, "gelu"), (nn.ReLU, "relu"), (nn.Identity, "identity")):
        if activation is cls or isinstance(activation, cls):
            return name
    raise ValueError(f"unsupported activation {activation!r}; expected nn.ReLU, nn.SiLU, nn.GELU or nn.Identity")


def _versions(module: nn.Module) -> Tuple:
    return tuple((t.data_ptr(), t._version) for t in list(module.parameters()) + list(module.buffers()))


class _EngineCache:
    """Packed-weight cache: rebuilt when any parameter is replaced or modified in place
    (optimizer.step(), load_state_dict) or the precision / device changes."""

    def __init__(self) -> None:
        self.key = None
        self.value = None

    def get(self, module: nn.Module, precision: str, build):
        dev = next(module.parameters()).device
        key = (precision, str(dev), _versions(module))
        if key != self.key:
            self.value = build(dev)
            self.key = key
        return self.value


def _require_cuda(t: torch.Tensor, what: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(f"{what}: parameters are on {t.device}; sbgm_danra_b200 has no CPU path -- move the model to a CUDA device")


class SinusoidalEmbedding(nn.Module):
    """Gaussian-Fourier time features: cat(sin(2 pi t W), cos(2 pi t W)), W fixed (score_unet.py:24-45)."""

    def __init__(self, embed_dim: int, scale: float = 30.0, device=None, dtype=torch.float32):
        super().__init__()
        if embed_dim % 2 != 0:
            raise ValueError(f"Embedding dimension must be even, got {embed_dim}.")
        self.register_buffer("W", torch.randn(embed_dim // 2, dtype=dtype, device=device) * scale, persistent=True)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        _require_cuda(self.W, "SinusoidalEmbedding")
        t = x.reshape(-1).to(device=self.W.device, dtype=torch.float32).contiguous()
        w = self.W.float().contiguous()
        out = torch.empty((t.numel(), 2 * w.numel()), dtype=torch.float32, device=w.device)
        with torch.cuda.device(w.device):
            call("sbgm_fourier_embed", t.data_ptr(), w.data_ptr(), w.numel(), out.data_ptr(), t.numel(), _eng._stream())
        return out


class ImageSelfAttention(nn.Module):
    """Pre-LayerNorm self-attention + feed-forward over flattened pixels (score_unet.py:112-148)."""

    def __init__(self, input_channels: int, n_heads: int, dropout: float = 0.0):
        super().__init__()
        if input_channels % n_heads != 0:
            raise ValueError(f"Number of input channels ({input_channels}) must be divisible by number of heads ({n_heads}).")
        if dropout != 0.0:
            raise NotImplementedError("attention dropout is not on the CUDA path (the reference never enables it)")
        self.input_channels, self.n_heads = input_channels, n_heads
        self.mha = nn.MultiheadAttention(embed_dim=input_channels, num_heads=n_heads, dropout=dropout, batch_first=True)
        self.ln1 = nn.LayerNorm(input_channels)
        self.ln2 = nn.LayerNorm(input_channels)
        self.ff = nn.Sequential(nn.Linear(input_channels, input_channels), nn.GELU(), nn.Linear(input_channels, input_channels))
        self.precision = DEFAULT_PRECISION
        self._cache = _EngineCache()

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        _require_cuda(self.ln1.weight, "ImageSelfAttention")

        def build(dev):
            fmt = _eng.PRECISIONS[self.precision]
            return _eng.Kernels(fmt, dev), _eng.AttentionW(_eng._Packer(self.state_dict(), fmt, dev), _eng.attention_layout(""),
                                                           self.n_heads), fmt

        with torch.no_grad(), torch.cuda.device(self.ln1.weight.device):
            k, aw, fmt = self._cache.get(self, self.precision, build)
            a = _eng.Act.from_nchw(x.to(self.ln1.weight.device), fmt)
            return _eng.attention_block(k, aw, a).to_nchw()


class _ResidualBlock(nn.Module):
    """Parameter container for a torchvision-style BasicBlock (resnet.py:59-103): same child names."""
    expansion = 1

    def __init__(self, inplanes: int, planes: int, stride: int):
        super().__init__()
        self.conv1 = nn.Conv2d(inplanes, planes, 3, stride, 1, bias=False)
        self.bn1 = nn.BatchNorm2d(planes)
        self.conv2 = nn.Conv2d(planes, planes, 3, 1, 1, bias=False)
        self.bn2 = nn.BatchNorm2d(planes)
        self.downsample = None
        if stride != 1 or inplanes != planes:
            self.downsample = nn.Sequential(nn.Conv2d(inplanes, planes, 1, stride, bias=False), nn.BatchNorm2d(planes))
        self.stride = stride
        for m in (self.conv1, self.conv2) + ((self.downsample[0],) if self.downsample is not None else ()):
            nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="relu")


def _resolve_block(block) -> None:
    name = getattr(block, "__name__", str(block))
    if block is not None and name != "BasicBlock" and block is not _ResidualBlock:
        raise NotImplementedError(f"Encoder block {name}: only the BasicBlock topology is on the CUDA path")


class Encoder(nn.Module):
    """ResNet-style conditional encoder producing five skip feature maps (score_unet.py:151-397)."""

    def __init__(self, input_channels: int, time_embedding: int, block=None, block_layers: list = [2, 2, 2, 2],
                 n_heads: int = 4, num_classes: Optional[int] = None, cond_on_img=False, cond_img_dim=None, device=None):
        super().__init__()
        _resolve_block(block)
        if len(block_layers) != 4:
            raise ValueError(f"block_layers must have 4 entries, got {block_layers}")
        self.block_layers = list(block_layers)
        self.time_embedding = time_embedding
        self.input_channels = input_channels + 1   # + the noised HR field
        self.n_heads = n_heads
        self.num_classes = num_classes
        self.device = _default_device(device)
        self.conv1 = nn.Conv2d(self.input_channels, 64, kernel_size=(8, 8), stride=(2, 2), padding=(3, 3), bias=False)
        self.bn1 = nn.BatchNorm2d(64)
        inplanes = 64
        for li, (planes, nblk) in enumerate(zip((64, 128, 256, 512), self.block_layers), start=1):
            blocks = []
            for b in range(nblk):
                blocks.append(_ResidualBlock(inplanes, planes, 2 if (b == 0 and li > 1) else 1))
                inplanes = planes
            setattr(self, f"layer{li}", nn.Sequential(*blocks))
        self.sinusoidal_embedding = SinusoidalEmbedding(time_embedding)
        self.time_projection_layers = self.make_time_projections(_eng.FMAP_CHANNELS)
        self.attention_layers = self.make_attention_layers(_eng.FMAP_CHANNELS)
        self.conv2 = nn.Conv2d(64, 64, kernel_size=(8, 8), stride=(2, 2), padding=(3, 3), bias=False)
        if num_classes is not None:
            self.label_emb = nn.Embedding(num_classes + 1, time_embedding)
            with torch.no_grad():
                self.label_emb.weight[0].fill_(0.0)   # null class (classifier-free guidance)
        self.precision = DEFAULT_PRECISION
        self._cache = _EngineCache()

    def make_time_projections(self, fmap_channels: Iterable[int]) -> nn.ModuleList:
        return nn.ModuleList([nn.Sequential(nn.SiLU(), nn.Linear(self.time_embedding, ch)) for ch in fmap_channels])

    def make_attention_layers(self, fmap_channels: Iterable[int]) -> nn.ModuleList:
        chans = list(fmap_channels)
        return nn.ModuleList([ImageSelfAttention(ch, self.n_heads) if i >= len(chans) - 2 else nn.Identity()
                              for i, ch in enumerate(chans)])

    def _spec(self) -> _eng.UNetSpec:                       # the encoder's fields (the decoder's keep their defaults, unread)
        return _eng.UNetSpec(time_embedding=self.time_embedding, block_layers=tuple(self.block_layers), n_heads=self.n_heads,
                             has_labels=self.num_classes is not None)

    def _engine(self):
        def build(dev):
            tp = _eng.TimeProjector(dev, self.time_embedding)
            spec = self._spec()
            enc = _eng.EncoderEngine(self.state_dict(), spec, _eng.encoder_layout(spec, ""), fmt=_eng.PRECISIONS[self.precision],
                                     device=dev, tp=tp)
            tp.finalize()
            return enc
        return self._cache.get(self, self.precision, build)

    def forward(self, x: torch.Tensor, t: torch.Tensor, y: Optional[torch.Tensor] = None,
                cond_img: Optional[torch.Tensor] = None, lsm_cond: Optional[torch.Tensor] = None,
                topo_cond: Optional[torch.Tensor] = None):
        _require_cuda(self.conv1.weight, "Encoder")
        dev = self.conv1.weight.device
        if self.training and any(isinstance(m, nn.BatchNorm2d) for m in self.modules()):
            # .train(): batch statistics, running statistics and num_batches_tracked updated as nn.BatchNorm2d does (the
            # reference's Encoder.forward, score_unet.py:247-364, in training mode).  The standalone call returns detached
            # feature maps; gradients flow through ScoreNet.forward / loss_fn, which own the backward tape.
            from .train_engine import TrainEngine
            with torch.no_grad(), torch.cuda.device(dev):
                tensors = dict(list(self.named_parameters()) + list(self.named_buffers()))
                eng = TrainEngine(tensors, self._spec(), self.precision, dev, bn_train=True, encoder_only=True)
                planes = _eng.concat_planes(x.shape[0], lsm_cond, topo_cond, cond_img, dev)
                if planes is not None and planes.shape[0] != x.shape[0]:
                    planes = planes.expand(x.shape[0], -1, -1, -1).contiguous()
                fmaps = eng.forward(x.to(device=dev, dtype=torch.float32).contiguous(), t.to(dev), None if y is None else y.to(dev),
                                    planes, None)
                for m in self.modules():
                    if isinstance(m, nn.BatchNorm2d) and m.num_batches_tracked is not None:
                        m.num_batches_tracked += 1
                return tuple(f.to_nchw() for f in fmaps)
        with torch.no_grad(), torch.cuda.device(dev):
            enc = self._engine()
            x = x.to(device=dev, dtype=torch.float32).contiguous()
            planes = _eng.concat_planes(x.shape[0], lsm_cond, topo_cond, cond_img, dev)
            tproj = enc.tp(t.to(dev), None if y is None else y.to(dev))
            return tuple(f.to_nchw() for f in enc.forward(x, planes, tproj))


class DecoderBlock(nn.Module):
    """Upsample x2 -> conv -> norm -> conv -> norm -> +skip -> +time -> activation -> attention
    (score_unet.py:409-627)."""

    def __init__(self, input_channels: int, output_channels: int, time_embedding: int, upsample_scale: int = 2,
                 activation=nn.ReLU, compute_attn: bool = True, n_heads: int = 4, device=None, *,
                 use_resize_conv: bool = True, norm: str = "instance", gn_groups: int = 8):
        super().__init__()
        if upsample_scale != 2:
            raise NotImplementedError("only upsample_scale=2 is on the CUDA path (the reference never uses another)")
        self.device = _default_device(device)
        self.input_channels, self.output_channels = input_channels, output_channels
        self.upsample_scale, self.time_embedding = upsample_scale, time_embedding
        self.compute_attn, self.n_heads = compute_attn, n_heads
        self.use_resize_conv, self.norm_kind, self.gn_groups = use_resize_conv, norm, gn_groups
        if use_resize_conv:
            self.upsample = nn.Upsample(scale_factor=upsample_scale, mode="bilinear", align_corners=False)
            self.conv_up = nn.Conv2d(input_channels, input_channels, kernel_size=3, padding=1, bias=True)
        else:
            self.transpose = nn.ConvTranspose2d(input_channels, input_channels, kernel_size=upsample_scale, stride=upsample_scale)
        self.norm1 = self._make_norm(input_channels)
        self.conv = nn.Conv2d(input_channels, output_channels, kernel_size=3, padding=1)
        self.norm2 = self._make_norm(output_channels)
        self.activation = activation()
        self.sinusoidal_embedding = SinusoidalEmbedding(time_embedding)
        self.time_projection_layer = nn.Sequential(nn.SiLU(), nn.Linear(time_embedding, output_channels))
        self.attention = ImageSelfAttention(output_channels, n_heads) if compute_attn else nn.Identity()
        self.precision = DEFAULT_PRECISION
        self._cache = _EngineCache()

    def _make_norm(self, c: int) -> nn.Module:
        if self.norm_kind == "group":
            return nn.GroupNorm(num_groups=max(1, min(self.gn_groups, c)), num_channels=c)
        return nn.InstanceNorm2d(c)

    def forward(self, fmap: torch.Tensor, prev_fmap: Optional[torch.Tensor] = None, t: Optional[torch.Tensor] = None):
        """Standalone block evaluation (the fused ScoreNet path does not go through here)."""
        n1, n2 = getattr(self, "norm1", None), getattr(self, "norm2", None)
        if n1 is None or n2 is None:
            raise ValueError("Norm layers not found; possible init error.")
        _require_cuda(self.conv.weight, "DecoderBlock")
        id1, id2 = isinstance(n1, nn.Identity), isinstance(n2, nn.Identity)
        dev = self.conv.weight.device

        def build(d):
            fmt = _eng.PRECISIONS[self.precision]
            pk = _eng._Packer(self.state_dict(), fmt, d)
            s = _eng.decoder_block_layout("", "dec0", self.input_channels, self.output_channels, self.compute_attn, self.norm_kind,
                                          self.gn_groups, self.use_resize_conv)
            s = s._replace(n1=None if id1 else s.n1, n2=None if id2 else s.n2)      # an Identity norm (Decoder.final_layer) has no keys
            tp = _eng.TimeProjector(d, self.time_embedding)
            tp.add_heads([s.head], pk.get)
            tp.finalize()
            blk = _eng.pack_decoder_block(pk, s, self.use_resize_conv, self.n_heads)
            return _eng.Kernels(fmt, d), blk, tp, pk.conv(s.head.weight, s.head.bias), fmt

        with torch.no_grad(), torch.cuda.device(dev):
            k, blk, tp, tlin, fmt = self._cache.get(self, (self.precision, id1, id2), build)
            act = _eng.ACTS[_act_name(self.activation)]
            out_shape = (fmap.shape[0], self.output_channels, 2 * fmap.shape[2], 2 * fmap.shape[3])
            skip = None
            if prev_fmap is not None and torch.is_tensor(prev_fmap):
                if tuple(prev_fmap.shape) != out_shape:
                    raise AssertionError(f"prev_fmap shape {tuple(prev_fmap.shape)} must match output shape {out_shape}")
                skip = _eng.Act.from_nchw(prev_fmap.to(dev), fmt)
            tcols = None
            if t is not None:
                t = t.to(dev)
                if t.dim() == 1 or (t.dim() == 2 and t.shape[-1] != self.time_embedding):      # raw timesteps [B]
                    tcols = tp.cols(tp(t.reshape(-1).float(), None), blk.head.name)
                else:                                   # a precomputed embedding [B, time_dim]: SiLU -> Linear on the kernels
                    tcols = self._project_embedding(k, tlin, t.float(), fmt)
            x = _eng.Act.from_nchw(fmap.to(dev), fmt)
            a = k.conv(k.upsample2x(x), blk.conv_up, pad=1) if self.use_resize_conv else k.conv_transpose2x(x, blk.conv_up)
            if not id1:
                a = k.groupnorm(a, *blk.n1, groups=blk.g1)
            b = k.conv(a, blk.conv, pad=1)
            if id2:
                out = k.affine(b, skip=skip, tproj=tcols, act=act)            # x + prev_fmap + t_proj, then the activation
            else:
                out = k.groupnorm(b, *blk.n2, groups=blk.g2, act=act, skip=skip, tproj=tcols)
            if blk.attn is not None:
                out = _eng.attention_block(k, blk.attn, out)
            return out.to_nchw()

    def _project_embedding(self, k, lin: _eng.ConvW, t_emb: torch.Tensor, fmt: int) -> torch.Tensor:
        """time_projection_layer (SiLU -> `lin`, its packed Linear) of a precomputed embedding [B, time_dim] -> fp32 [B, C_out]."""
        rows = t_emb.shape[0]
        tok = _eng.Act.from_nchw(t_emb.t().reshape(1, self.time_embedding, 1, rows).contiguous(), fmt)
        h = tok.like()
        _eng.call("sbgm_act_forward", tok.ptr, tok.plane, h.ptr, h.plane, fmt, tok.plane, _eng.ACTS["silu"], _eng._stream())
        out = k.linear(h, lin)
        return out.to_nchw().reshape(self.output_channels, rows).t().contiguous()


class Decoder(nn.Module):
    """Four residual up-blocks with skip connections plus the final projection (score_unet.py:662-789)."""

    def __init__(self, last_fmap_channels: int, output_channels: int, time_embedding: int, first_fmap_channels: int = 64,
                 n_heads: int = 4, device=None, *, use_resize_conv: bool = True, norm: str = "instance",
                 gn_groups: int = 8, activation=nn.ReLU):
        super().__init__()
        self.device = _default_device(device)
        self.last_fmap_channels, self.output_channels = last_fmap_channels, output_channels
        self.time_embedding, self.first_fmap_channels, self.n_heads = time_embedding, first_fmap_channels, n_heads
        self.use_resize_conv, self.norm, self.gn_groups, self.activation = use_resize_conv, norm, gn_groups, activation
        self.residual_layers = self.make_layers()
        self.final_layer = DecoderBlock(self.residual_layers[-1].input_channels, output_channels, time_embedding=time_embedding,
                                        activation=nn.Identity, compute_attn=False, n_heads=n_heads, device=self.device,
                                        use_resize_conv=use_resize_conv, norm=norm, gn_groups=gn_groups)
        # the last block has neither norms nor activation (score_unet.py:726-730)
        self.final_layer.norm1 = nn.Identity()
        self.final_layer.norm2 = nn.Identity()
        self.final_layer.activation = nn.Identity()
        self.precision = DEFAULT_PRECISION
        self._cache = _EngineCache()

    def make_layers(self, n: int = 4) -> nn.ModuleList:
        layers: List[DecoderBlock] = []
        for i in range(n):
            in_ch = self.last_fmap_channels if i == 0 else layers[i - 1].output_channels
            out_ch = in_ch // 2 if i != (n - 1) else self.first_fmap_channels
            layers.append(DecoderBlock(in_ch, out_ch, time_embedding=self.time_embedding, compute_attn=(i < 2),
                                       n_heads=self.n_heads, device=self.device, use_resize_conv=self.use_resize_conv,
                                       norm=self.norm, gn_groups=self.gn_groups, activation=self.activation))
        return nn.ModuleList(layers)

    def plan(self) -> Tuple[Tuple[int, int, bool], ...]:
        return tuple((b.input_channels, b.output_channels, b.compute_attn) for b in self.residual_layers)

    def _engine(self):
        def build(dev):
            fmt = _eng.PRECISIONS[self.precision]
            tp = _eng.TimeProjector(dev, self.time_embedding)
            spec = _eng.UNetSpec(time_embedding=self.time_embedding, n_heads=self.n_heads, plan=self.plan(),
                                 out_channels=self.output_channels, use_resize_conv=self.use_resize_conv, norm=self.norm,
                                 gn_groups=self.gn_groups, activation=_act_name(self.activation))
            dec = _eng.DecoderEngine(self.state_dict(), spec, _eng.decoder_layout(spec, ""), fmt=fmt, device=dev, tp=tp)
            tp.finalize()
            return dec, fmt
        return self._cache.get(self, self.precision, build)

    def forward(self, *fmaps, t: Optional[torch.Tensor] = None):
        assert len(fmaps) == len(self.residual_layers) + 1, \
            f"Decoder expected {len(self.residual_layers) + 1} feature maps, got {len(fmaps)}"
        if t is None:
            raise ValueError("Decoder.forward needs the time tensor t")
        _require_cuda(self.final_layer.conv.weight, "Decoder")
        dev = self.final_layer.conv.weight.device
        with torch.no_grad(), torch.cuda.device(dev):
            dec, fmt = self._engine()
            acts = [_eng.Act.from_nchw(f.to(dev), fmt) for f in fmaps]
            tproj = dec.tp(t.to(dev), None)
            return dec.forward(acts, tproj, _eng.InvStd(None))


class ScoreNet(nn.Module):
    """score(x, t | conditions) = Decoder(Encoder(x, t, conditions)) / marginal_prob_std(t)
    (score_unet.py:792-879).  `precision` selects the kernel arithmetic (see engine.py)."""

    def __init__(self, marginal_prob_std, encoder: nn.Module, decoder: nn.Module, device=None,
                 debug_pre_sigma_div: bool = True):
        super().__init__()
        self.device = _default_device(device)
        self.marginal_prob_std = marginal_prob_std
        self.encoder = encoder
        self.decoder = decoder
        self.debug_pre_sigma_div = debug_pre_sigma_div
        self.precision = DEFAULT_PRECISION
        self._cache = _EngineCache()
        self.to(self.device)

    def spec(self) -> _eng.UNetSpec:
        e, d = self.encoder, self.decoder
        return _eng.UNetSpec(time_embedding=e.time_embedding, block_layers=tuple(e.block_layers), n_heads=e.n_heads,
                             has_labels=e.num_classes is not None, plan=d.plan(), out_channels=d.output_channels,
                             use_resize_conv=d.use_resize_conv, norm=d.norm, gn_groups=d.gn_groups, activation=_act_name(d.activation))

    def engine(self) -> _eng.UNetEngine:
        """Packed-weight engine for the current parameters (cached; rebuilt after parameter updates)."""
        _require_cuda(self.encoder.conv1.weight, "ScoreNet")
        return self._cache.get(self, self.precision, lambda dev: _eng.UNetEngine(self.state_dict(), self.spec(), self.precision, dev))

    # derived device state (packed weights, captured CUDA graphs, gradient exchange): never copied or pickled with the model
    _DERIVED = ("_cache", "_train_runners", "_grad_sync", "_members")

    def __deepcopy__(self, memo):
        """`copy.deepcopy(model)` (the reference's EMA copy, sbgm/training.py:114) copies parameters and buffers only; the copy
        builds its own engines on first use."""
        import copy
        new = self.__class__.__new__(self.__class__)
        memo[id(self)] = new
        for k, v in self.__dict__.items():
            if k not in self._DERIVED:
                new.__dict__[k] = copy.deepcopy(v, memo)
        new.__dict__["_cache"] = _EngineCache()
        return new

    def __getstate__(self):
        return {k: v for k, v in self.__dict__.items() if k not in self._DERIVED}

    def __setstate__(self, state):
        super().__setstate__(state)
        self.__dict__["_cache"] = _EngineCache()

    def _bn_modules(self):
        return self._member_lists()[3]

    def _member_lists(self):
        """(parameter names, parameters, named buffers, BatchNorm modules) of the module tree, cached: four traversals of
        ~120 modules cost ~0.5 ms of host time per training step, during which the GPU of a loop that reads `loss.item()`
        every step (sbgm/training.py:410) sits idle.  The cache is dropped by `_apply` (.to / .cuda / .float) and checked
        against the identity of the first and last parameter and buffer; code that swaps a parameter or a submodule in the
        middle of the tree after the first training forward must call `model.invalidate_members()`."""
        m = self.__dict__.get("_members")
        if m is not None:
            names, params, buffers, _ = m
            first, last = names[0], names[-1]
            if (self.get_parameter(first) is params[0] and self.get_parameter(last) is params[-1]
                    and (not buffers or self.get_buffer(buffers[-1][0]) is buffers[-1][1])):
                return m
        named = list(self.named_parameters())
        m = ([k for k, _ in named], [p for _, p in named], list(self.named_buffers()),
             [mod for mod in self.modules() if isinstance(mod, nn.BatchNorm2d)])
        self.__dict__["_members"] = m
        return m

    def invalidate_members(self) -> None:
        self.__dict__.pop("_members", None)

    def _apply(self, fn, *args, **kwargs):
        self.__dict__.pop("_members", None)
        return super()._apply(fn, *args, **kwargs)

    def load_state_dict(self, *args, **kwargs):
        self.__dict__.pop("_members", None)
        return super().load_state_dict(*args, **kwargs)

    def forward(self, x: torch.Tensor, t: torch.Tensor, y: Optional[torch.Tensor] = None,
                cond_img: Optional[torch.Tensor] = None, lsm_cond: Optional[torch.Tensor] = None,
                topo_cond: Optional[torch.Tensor] = None) -> torch.Tensor:
        _require_cuda(self.encoder.conv1.weight, "ScoreNet")
        dev = self.encoder.conv1.weight.device
        needs_grad = False
        if torch.is_grad_enabled() or self.training:
            names, params, _, bn_modules = self._member_lists()
            # the differentiable path also when only inputs want a gradient (a frozen model under torch.autograd.grad)
            needs_grad = torch.is_grad_enabled() and (any(p.requires_grad for p in params) or any(
                v is not None and v.requires_grad for v in (x, cond_img, lsm_cond, topo_cond)))
        if needs_grad or self.training:
            # training graph: unfolded BatchNorm (batch statistics when .training), backward tape (train_engine.py)
            with torch.cuda.device(dev):
                x = x.to(dev).float().contiguous()
                t = t.to(dev).float()
                planes = _eng.concat_planes(x.shape[0], lsm_cond, topo_cond, cond_img, dev)
                std = self.marginal_prob_std(t)
                pre = bool(getattr(self, "debug_pre_sigma_div", True))
                inv_std = None if pre else (1.0 / std.float()).contiguous()
                out = _ScoreNetFn.apply(self, x, t, y, planes, inv_std, names, torch.is_grad_enabled(), *params)
                if self.training:
                    torch._foreach_add_([m.num_batches_tracked for m in bn_modules], 1)
                if pre:
                    with torch.no_grad():
                        logger.info(f"[pre-σ-div] mean = {float(out.mean()):.4g}, std = {float(out.std()):.4g}, "
                                    f"σ ∈ [{std.min():.4g}, {std.max():.4g}]")
                    return out / std.view(-1, 1, 1, 1)
                return out
        eng = self.engine()
        with torch.no_grad(), torch.cuda.device(dev):
            x = x.to(dev)
            t = t.to(dev).float()
            planes = _eng.concat_planes(x.shape[0], lsm_cond, topo_cond, cond_img, dev)
            std = self.marginal_prob_std(t)
            if getattr(self, "debug_pre_sigma_div", True):
                out = eng.forward(x, t, y, planes, None)
                logger.info(f"[pre-σ-div] mean = {float(out.mean()):.4g}, std = {float(out.std()):.4g}, "
                            f"σ ∈ [{std.min():.4g}, {std.max():.4g}]")
                return out / std.view(-1, 1, 1, 1)
            inv_std = (1.0 / std.float()).contiguous()
            return eng.forward(x, t, y, planes, inv_std)


def _detach_grads_aliasing(params, flat) -> None:
    """Give every `.grad` that is still a view of the engine's flat gradient buffer its own storage (the engine is about to
    overwrite the buffer: the captured forward re-zeroes it, backward refills it)."""
    if flat is None:
        return
    ptr = flat.untyped_storage().data_ptr()
    with torch.no_grad():
        for p in params:
            g = p.grad
            if g is not None and g.untyped_storage().data_ptr() == ptr:
                p.grad = g.clone()


class _ScoreNetFn(torch.autograd.Function):
    """The whole score-UNet as one autograd node: forward and backward both run this repo's kernels
    (train_engine.TrainEngine); replaces torch autograd over sbgm/score_unet.py:829-879."""

    @staticmethod
    def forward(ctx, model, x, t, y, planes, inv_std, names, grad_mode, *params):
        from .train_engine import TrainEngine, TrainRunner
        buffers = model._member_lists()[2]
        sync = getattr(model, "_grad_sync", None)
        # the captured graphs bake in the gradient exchange: a runner belongs to one GradSync object (parallel.attach / detach)
        sync_key = None if sync is None else (id(sync), bool(sync.sync_bn), sync.world)
        # which gradients backward produces: (x, planes) and whether the parameters' (all of them as soon as one wants one)
        input_grads = (grad_mode and ctx.needs_input_grad[1], grad_mode and ctx.needs_input_grad[4])
        param_grads = any(ctx.needs_input_grad[8:]) or not any(input_grads)
        key = (model.precision, model.training, tuple(x.shape), None if planes is None else tuple(planes.shape), y is None,
               inv_std is None, str(x.device), tuple(p.data_ptr() for p in params), tuple(b.data_ptr() for _, b in buffers), sync_key,
               input_grads, param_grads)
        runners = model.__dict__.setdefault("_train_runners", {})
        runner = runners.get(key)
        if runner is None:
            # the closure holds the model's tensors and settings, not the model: model -> runner -> closure -> model would be a
            # reference cycle, and the runner's CUDA graphs would then die whenever the cyclic collector runs (possibly inside
            # someone else's graph capture) instead of with the model
            spec, precision, training, device = model.spec(), model.precision, model.training, x.device

            def make_engine():
                tensors = dict(zip(names, params))
                tensors.update(buffers)
                return TrainEngine(tensors, spec, precision, device, bn_train=training, input_grads=input_grads, param_grads=param_grads)
            runners.clear()                       # one live configuration at a time (the graphs pin GBs of activations)
            runner = runners[key] = TrainRunner(make_engine, use_graphs=os.environ.get("SBGM_B200_TRAIN_GRAPHS", "1") != "0")
        if runner.eng is not None:                # captured step: its forward graph re-zeroes the flat gradient buffer
            _detach_grads_aliasing(params, runner.eng.flat)
        yy = None if y is None else y.reshape(-1).to(device=x.device, dtype=torch.int64).contiguous()
        out, handle = runner.forward(x, t.reshape(-1).float().contiguous(), yy, planes, inv_std, sync)
        ctx.runner, ctx.handle, ctx.names, ctx.params = runner, handle, names, params
        return out

    @staticmethod
    def backward(ctx, dout):
        runner, handle = ctx.runner, ctx.handle
        # Every parameter gradient is a view of the engine's flat buffer.  Returned as FRESH view objects (nothing else holds
        # them), autograd's AccumulateGrad adopts them as `.grad` instead of cloning 164 tensors per step (DDP's
        # gradient_as_bucket_view).  A `.grad` that still aliases the buffer from an earlier step (gradient accumulation,
        # zero_grad(set_to_none=False)) is detached into its own storage before the buffer is overwritten (here and in forward).
        # SBGM_B200_GRAD_VIEWS=0 restores independent `.grad` tensors (a held reference to an old `.grad` then survives the
        # next backward, at the price of the copies).
        views = os.environ.get("SBGM_B200_GRAD_VIEWS", "1") != "0"
        _detach_grads_aliasing(ctx.params, runner.flat_of(handle))
        with torch.cuda.device(dout.device):
            grads = runner.backward(handle, dout)
        names = ctx.names
        ctx.runner = ctx.handle = ctx.params = None
        out = []
        for n in names:
            g = grads.get(n)
            out.append(None if g is None else (g.view(g.shape) if views else g))
        from .train_engine import DPLANES, DX
        return (None, grads.get(DX), None, None, grads.get(DPLANES), None, None, None) + tuple(out)


class _DSMLossFn(torch.autograd.Function):
    """loss = mean_n sum_pix w (score std + z)^2 and its gradient w.r.t. score (score_unet.py:936-985)."""

    @staticmethod
    def forward(ctx, score, std, z, sdf):
        from . import _lib
        n, per = score.shape[0], score[0].numel()
        score = score.contiguous().float()
        partials = torch.empty(_lib.query("sbgm_dsm_scratch_floats", score.numel()), dtype=torch.float32, device=score.device)
        loss = torch.empty((), dtype=torch.float32, device=score.device)
        call("sbgm_dsm_loss", score.data_ptr(), std.data_ptr(), z.data_ptr(), None if sdf is None else sdf.data_ptr(),
             n, per, partials.data_ptr(), loss.data_ptr(), _eng._stream())
        ctx.save_for_backward(score, std, z, *(() if sdf is None else (sdf,)))
        return loss

    @staticmethod
    def backward(ctx, grad_loss):
        score, std, z, *rest = ctx.saved_tensors
        sdf = rest[0] if rest else None
        n, per = score.shape[0], score[0].numel()
        dscore = torch.empty_like(score)
        gl = grad_loss.to(device=score.device, dtype=torch.float32).contiguous()
        with torch.cuda.device(score.device):
            call("sbgm_dsm_loss_backward", score.data_ptr(), std.data_ptr(), z.data_ptr(), None if sdf is None else sdf.data_ptr(),
                 gl.data_ptr(), n, per, dscore.data_ptr(), _eng._stream())
        return dscore, None, None, None


def marginal_prob_std(t: torch.Tensor, sigma: float, eps: float = 1e-5) -> torch.Tensor:
    """VE-SDE marginal std sqrt((sigma^(2t) - 1) / (2 ln sigma)), clamped at eps (score_unet.py:881-897).
    A [B]-sized scalar schedule: evaluated with torch on whatever device `t` lives on."""
    t = t.to(dtype=torch.float32)
    key = (float(sigma), t.device)
    log_sigma = _LOG_SIGMA.get(key)
    if log_sigma is None:           # torch.tensor(..., device=cuda) is a blocking host-to-device copy: made once, not every call
        log_sigma = _LOG_SIGMA[key] = torch.log(torch.tensor(sigma, dtype=torch.float32, device=t.device))
    return torch.clamp(torch.sqrt((torch.exp((2.0 * t) * log_sigma) - 1.0) / (2.0 * log_sigma)), min=eps)


_LOG_SIGMA: dict = {}


def diffusion_coeff(t, sigma, device=None):
    """g(t) = sigma^t (score_unet.py:916-930)."""
    return (sigma ** t).to(t.device)


sigma = 25.0
marginal_prob_std_fn = functools.partial(marginal_prob_std, sigma=sigma)
diffusion_coeff_fn = functools.partial(diffusion_coeff, sigma=sigma)


def loss_fn(model, x, marginal_prob_std, t_eps=1e-3, device=None, y=None, cond_img=None, lsm_cond=None,
            topo_cond=None, sdf_cond=None):
    """Denoising score-matching loss (score_unet.py:936-985).

    t ~ U(t_eps, 1), z ~ N(0, I) come from the Philox stream of `sbgm_danra_b200.score_sampling.noise_state()`.
    With grad enabled the returned 0-d tensor carries an autograd graph whose nodes (`_DSMLossFn`, `_ScoreNetFn`)
    run this repo's backward kernels, so `loss.backward()` fills `param.grad` exactly as in the reference flow
    (sbgm/training.py:323-410)."""
    from . import score_sampling as _ss
    for name, arr in (("cond_img", cond_img), ("lsm_cond", lsm_cond), ("topo_cond", topo_cond), ("y", y)):
        if arr is not None and arr.shape[0] != x.shape[0]:
            raise ValueError(f"Batch size mismatch: x={x.shape[0]}, {name}={arr.shape[0]}")
    return _ss._dsm_loss_forward(model, x, marginal_prob_std, t_eps, y, cond_img, lsm_cond, topo_cond, sdf_cond)
