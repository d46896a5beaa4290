"""Kernel-level execution engine for the score-UNet: weight packing + the launch sequence.

The engine owns *derived* copies of the module parameters (NHWC / K-major, BatchNorm folded,
bf16 or split-bf16) and sequences the C-ABI kernels of `include/sbgm_b200.h` for one forward pass
(reference: Encoder.forward sbgm/score_unet.py:247-364, DecoderBlock.forward :559-627,
Decoder.forward :733-758, ScoreNet.forward :829-879).  torch is used for device memory and
streams only; every FLOP on the path runs in this repo's kernels.

Precisions
    "fp32"    exact fp32 arithmetic on CUDA cores (debug / strict-parity mode)
    "bf16x3"  tensor cores, split-bf16 operands (hi*hi + lo*hi + hi*lo), fp32 accumulate:
              fp32-class accuracy; this is the "fp32/TF32 mode" of the north star (plain TF32
              sits on the 1e-3 parity gate, SURVEY.md section 7)
    "bf16"    tensor cores, bf16 operands, fp32 accumulate
    "fp16x2"  tensor cores, ONE float16 activation plane, weights as float16 hi|lo planes (x*w_hi + x*w_lo: two
              products): the weights are exact to 22 bits, only the activations are rounded (11 bits) -- score
              rel-L2 2-5e-4 vs the reference's fp32, inside the 1e-3 gate -- at 2/3 of bf16x3's tensor work and
              half its activation bytes.  Inference only (training with it runs the bf16x3 kernels).
"""
from __future__ import annotations

from collections import namedtuple
from dataclasses import dataclass
from typing import Callable, Dict, List, NamedTuple, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import ACT_GELU, ACT_NONE, ACT_RELU, ACT_SILU, F16_WLO_SCALE, FMT_BF16, FMT_BF16X2, FMT_F16, FMT_F32, call

PRECISIONS = {"fp32": FMT_F32, "bf16x3": FMT_BF16X2, "bf16": FMT_BF16, "fp16x2": FMT_F16}
ACTS = {"relu": ACT_RELU, "silu": ACT_SILU, "gelu": ACT_GELU, "identity": ACT_NONE, None: ACT_NONE}
FMAP_CHANNELS = (64, 64, 128, 256, 512)
BN_EPS = 1e-5
GN_EPS = 1e-5
LN_EPS = 1e-5


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


# Timing ablations only (tools/ablate.py): SBGM_B200_SKIP=attn,attn_core,gn,ln,upsample,c64,conv_tc drops the named operator from
# the launch sequence so that its in-graph cost can be read off as a difference.  Results are garbage when set.
import os as _os
_SKIP = frozenset(x for x in _os.environ.get("SBGM_B200_SKIP", "").split(",") if x)


# Measurement hook (bench.py `roofline.family`): when set to a list, every convolution / Linear launch of a forward appends
# its geometry, so that the layers can afterwards be timed one by one.  None on the product path.
CONV_TRACE: Optional[list] = None


class Act:
    """An NHWC activation tensor in one of the four storage formats."""
    __slots__ = ("buf", "fmt", "n", "h", "w", "c")

    def __init__(self, fmt: int, n: int, h: int, w: int, c: int, device) -> None:
        self.fmt, self.n, self.h, self.w, self.c = fmt, n, h, w, c
        if fmt == FMT_F32:
            self.buf = torch.empty((n, h, w, c), dtype=torch.float32, device=device)
        elif fmt == FMT_BF16:
            self.buf = torch.empty((n, h, w, c), dtype=torch.bfloat16, device=device)
        elif fmt == FMT_F16:
            self.buf = torch.empty((n, h, w, c), dtype=torch.float16, device=device)
        else:
            self.buf = torch.empty((2, n, h, w, c), dtype=torch.bfloat16, device=device)

    @property
    def plane(self) -> int:
        return self.n * self.h * self.w * self.c

    @property
    def ptr(self) -> int:
        return self.buf.data_ptr()

    def view(self, n: int, h: int, w: int, c: int) -> "Act":
        """The same storage as an [n, h, w, c] tensor of the same size (no copy)."""
        v = Act.__new__(Act)
        v.buf, v.fmt, v.n, v.h, v.w, v.c = self.buf, self.fmt, n, h, w, c
        return v

    def tokens(self) -> "Act":
        """View [n, h, w, c] as a token matrix [1, 1, n*h*w, c] (no copy)."""
        return self.view(1, 1, self.n * self.h * self.w, self.c)

    def like(self, c: Optional[int] = None, h: Optional[int] = None, w: Optional[int] = None) -> "Act":
        return Act(self.fmt, self.n, h or self.h, w or self.w, c or self.c, self.buf.device)

    def to_nchw(self) -> torch.Tensor:
        out = torch.empty((self.n, self.c, self.h, self.w), dtype=torch.float32, device=self.buf.device)
        call("sbgm_nhwc_to_nchw", self.ptr, self.plane, self.fmt, out.data_ptr(), self.n, self.c, self.h, self.w, _stream())
        return out

    @staticmethod
    def from_nchw(x: torch.Tensor, fmt: int) -> "Act":
        x = x.contiguous().float()
        n, c, h, w = x.shape
        a = Act(fmt, n, h, w, c, x.device)
        call("sbgm_nchw_to_nhwc", x.data_ptr(), a.ptr, a.plane, fmt, n, c, h, w, _stream())
        return a


@dataclass
class ConvW:
    """A packed convolution / linear weight (+ folded bias)."""
    w: torch.Tensor
    bias: Optional[torch.Tensor]
    cin: int
    cout: int
    kh: int
    kw: int
    colsum: Optional[torch.Tensor] = None      # LayerNorm-folded Linear layers: row sums of the folded weight (fp32)

    @property
    def plane(self) -> int:
        return self.cout * self.kh * self.kw * self.cin


@dataclass
class TransposeW:
    """A packed nn.ConvTranspose2d(cin, cout, kernel 2, stride 2) (score_unet.py:466-468, the use_resize_conv=False decoder):
    out[n, 2i+a, 2j+b, co] = bias[co] + sum_ci x[n, i, j, ci] W[ci][co][a][b] -- four 1x1 convolutions scattered to the four
    output parities (`subs`: (a, b, ConvW), tensor cores), or one gather over the 2x2 taps (`simt` [4][cin][cout], fp32)."""
    bias: torch.Tensor
    cin: int
    cout: int
    simt: Optional[torch.Tensor] = None
    subs: Optional[List[Tuple[int, int, ConvW]]] = None


def pack_transpose(w: torch.Tensor, bias: torch.Tensor, fmt: int, pack_sub: Callable[[int, int], torch.Tensor]) -> TransposeW:
    """`w` [cin][cout][2][2] fp32; `pack_sub(a, b)`: the tensor-core storage of the K-major matrix w[:, :, a, b]^T."""
    cin, cout = w.shape[0], w.shape[1]
    if fmt == FMT_F32:
        return TransposeW(bias, cin, cout, simt=w.permute(2, 3, 0, 1).reshape(4, cin, cout).contiguous())
    return TransposeW(bias, cin, cout, subs=[(a, b, ConvW(pack_sub(a, b), bias, cin, cout, 1, 1)) for a in range(2) for b in range(2)])


class InvStd(NamedTuple):
    """Where the final layer reads 1/std: sample n of the current step takes values[n * stride + step * step_stride], with
    step = *step_counter (0 without a counter); no values: no scaling.  A sampler passes its step table's 1/std column, stride 0,
    the table's row length and the device step counter."""
    values: Optional[torch.Tensor]
    stride: int = 1
    step_stride: int = 0
    step_counter: Optional[torch.Tensor] = None

    def args(self) -> tuple:
        return _ptr(self.values), self.stride, self.step_stride, _ptr(self.step_counter)


def _split_bf16(x: torch.Tensor) -> torch.Tensor:
    hi = x.to(torch.bfloat16)
    lo = (x - hi.float()).to(torch.bfloat16)
    return torch.stack([hi, lo]).contiguous()


def _split_f16(x: torch.Tensor) -> torch.Tensor:
    """float16 hi | lo * 2^11 planes of a weight matrix (SBGM_FMT_F16 layers): 22 significant bits.  |w| beyond the float16
    range saturates (a BatchNorm-folded weight of 6e4 would be a broken checkpoint anyway)."""
    hi = x.clamp(-65504.0, 65504.0).to(torch.float16)
    lo = ((x - hi.float()) * F16_WLO_SCALE).to(torch.float16)
    return torch.stack([hi, lo]).contiguous()


def pack_tc_matrix(km: torch.Tensor, fmt: int) -> torch.Tensor:
    """K-major weight matrix [cout][K] fp32 -> the tensor-core storage of `fmt`."""
    if fmt == FMT_BF16:
        return km.to(torch.bfloat16)
    return _split_f16(km) if fmt == FMT_F16 else _split_bf16(km)


class _Packer:
    def __init__(self, sd: Dict[str, torch.Tensor], fmt: int, device) -> None:
        self.sd, self.fmt, self.device = sd, fmt, device

    def get(self, key: str) -> torch.Tensor:
        return self.sd[key].detach().to(device=self.device, dtype=torch.float32)

    def vec(self, key: str) -> torch.Tensor:
        return self.get(key).contiguous()

    def conv(self, wkey: str, bias_key: Optional[str] = None, bn=None) -> ConvW:
        w = self.get(wkey)
        if w.dim() == 2:
            w = w[:, :, None, None]
        cout, cin, kh, kw = w.shape
        bias = self.get(bias_key) if bias_key is not None else None
        if bn is not None:   # eval-mode BatchNorm folded into the convolution
            bn = batchnorm_keys(bn) if isinstance(bn, str) else bn      # the BatchNorm2d's key prefix or its BatchNormKeys
            scale = self.get(bn.weight) / torch.sqrt(self.get(bn.running_var) + BN_EPS)
            shift = self.get(bn.bias) - self.get(bn.running_mean) * scale
            w = w * scale[:, None, None, None]
            bias = shift if bias is None else bias * scale + shift
        if self.fmt == FMT_F32:
            packed = w.permute(2, 3, 1, 0).reshape(kh * kw * cin, cout).contiguous()      # [K][cout]
        else:
            km = w.permute(0, 2, 3, 1).reshape(cout, kh * kw * cin).contiguous()           # [cout][K]
            packed = pack_tc_matrix(km, self.fmt)
        return ConvW(packed, None if bias is None else bias.contiguous(), cin, cout, kh, kw)

    def conv_transpose(self, wkey: str, bias_key: str) -> TransposeW:
        w = self.get(wkey)                                    # [cin, cout, 2, 2]
        return pack_transpose(w, self.vec(bias_key), self.fmt, lambda a, b: pack_tc_matrix(w[:, :, a, b].t().contiguous(), self.fmt))

    def up(self, site: "Affine", resize: bool):          # a decoder up-path: resize convolution (ConvW) or transposed one (TransposeW)
        return self.conv(*site) if resize else self.conv_transpose(*site)


def _unpack_tc_matrix(packed: torch.Tensor, fmt: int) -> torch.Tensor:
    """The fp32 values a tensor-core layer actually multiplies with (inverse of pack_tc_matrix up to its rounding)."""
    if fmt == FMT_BF16:
        return packed.float()
    if fmt == FMT_F16:
        return packed[0].float() + packed[1].float() / F16_WLO_SCALE
    return packed[0].float() + packed[1].float()


def pack_linear_ln(pk: "_Packer", wkey: str, bkey: str, gkey: str, betakey: str) -> ConvW:
    """Linear layer behind a LayerNorm, folded (sbgm_linear_ln_tc): W' = W diag(gamma), b' = b + W beta, colsum = W' 1.
    The column sums are taken over the packed (rounded) weights, so that  x W'^T - mean colsum  cancels exactly as
    (x - mean) W'^T would."""
    w, b = pk.get(wkey), pk.get(bkey)
    gamma, beta = pk.get(gkey), pk.get(betakey)
    wf = (w * gamma[None, :]).contiguous()
    bf = (b + w @ beta).contiguous()
    packed = pack_tc_matrix(wf, pk.fmt)
    colsum = _unpack_tc_matrix(packed, pk.fmt).double().sum(dim=1).float().contiguous()
    return ConvW(packed, bf, w.shape[1], w.shape[0], 1, 1, colsum)


class Kernels:
    """Thin typed wrappers over the C ABI operating on `Act` tensors."""

    def __init__(self, fmt: int, device) -> None:
        self.fmt, self.device = fmt, device
        self._gn_scratch: Optional[torch.Tensor] = None
        self._splitk_ws: Optional[torch.Tensor] = None

    def _c64_ok(self, x: Act, cw: ConvW, stride: int, pad: int) -> bool:
        return (self.fmt != FMT_F32 and cw.cin == 64 and cw.cout == 64 and cw.kh == 3 and cw.kw == 3 and stride == 1
                and pad == 1 and x.h % 16 == 0 and x.w % 8 == 0)

    def conv(self, x: Act, cw: ConvW, stride: int = 1, pad: int = 0, act: int = ACT_NONE,
             residual: Optional[Act] = None, tproj: Optional[torch.Tensor] = None,
             proj: Optional[torch.Tensor] = None, gn_stats: bool = False, proj_keep: bool = False):
        """Convolution + fused epilogue.  Returns the output `Act`; with `proj` ([n_proj, 64] fp32) returns the
        projected fp32 tensor [n, h, w, PROJ_STRIDE] instead; with `gn_stats=True` returns (Act, stats) where
        stats = (partials, chunks) if the producing kernel could fuse the GroupNorm statistics, else None."""
        assert x.c == cw.cin, f"conv: input has {x.c} channels, weight expects {cw.cin}"
        if CONV_TRACE is not None:
            CONV_TRACE.append(dict(n=x.n, h=x.h, w=x.w, cw=cw, stride=stride, pad=pad, act=act, residual=residual is not None,
                                   tproj=tproj is not None, proj=proj is not None, gn_stats=gn_stats,
                                   c64=self._c64_ok(x, cw, stride, pad)))
        ho = (x.h + 2 * pad - cw.kh) // stride + 1
        wo = (x.w + 2 * pad - cw.kw) // stride + 1
        tp_ptr = _ptr(tproj)
        tp_stride = tproj.stride(0) if tproj is not None else 0
        res_ptr = None if residual is None else residual.ptr
        res_plane = 0 if residual is None else residual.plane
        if proj is not None:
            assert self.fmt != FMT_F32 and cw.cout == 64
            out, out_ptr, out_plane = None, None, 0
            if proj_keep:           # training: the projected tensor AND the convolution output (64 -> 64 kernel only)
                assert self._c64_ok(x, cw, stride, pad)
                out = Act(self.fmt, x.n, ho, wo, cw.cout, self.device)
                out_ptr, out_plane = out.ptr, out.plane
            pout = torch.empty((x.n, ho, wo, _lib.PROJ_STRIDE), dtype=torch.float32, device=self.device)
            pargs = (proj.data_ptr(), proj.shape[0], pout.data_ptr())
        else:
            out = Act(self.fmt, x.n, ho, wo, cw.cout, self.device)
            out_ptr, out_plane, pout, pargs = out.ptr, out.plane, None, (None, 0, None)
        stats = None
        skip_this = ("c64" in _SKIP and self._c64_ok(x, cw, stride, pad)) or ("conv_tc" in _SKIP and not self._c64_ok(x, cw, stride, pad))
        if _SKIP and not self._c64_ok(x, cw, stride, pad):      # finer classes of the generic kernel
            cls = "tc_1x1" if cw.kh == 1 else "tc_s2" if stride != 1 else "tc_big" if x.h >= 16 else "tc_8" if x.h == 8 else "tc_4"
            skip_this = skip_this or cls in _SKIP
        if skip_this:                      # timing ablation: leave the output uninitialised
            if proj is not None:
                return (out, pout) if proj_keep else pout
            return (out, None) if gn_stats else out
        if self.fmt == FMT_F32:
            call("sbgm_conv2d_simt", x.ptr, cw.w.data_ptr(), _ptr(cw.bias), res_ptr, tp_ptr, tp_stride, out.ptr,
                 x.n, x.h, x.w, cw.cin, cw.cout, cw.kh, cw.kw, stride, pad, act, _stream())
        elif self._c64_ok(x, cw, stride, pad):
            part = None
            if gn_stats and residual is None and tproj is None and act == ACT_NONE and proj is None:
                chunks = (x.h // 16) * (x.w // 8) * 4
                part = torch.empty((x.n, chunks, 8, 2), dtype=torch.float32, device=self.device)
                stats = (part, chunks)
            call("sbgm_conv3x3_c64", x.ptr, x.plane, cw.w.data_ptr(), cw.plane, _ptr(cw.bias), res_ptr, res_plane,
                 tp_ptr, tp_stride, out_ptr, out_plane, self.fmt, x.n, x.h, x.w, act, *pargs, _ptr(part), 8, _stream())
        else:
            ws_bytes = 0 if proj is not None else _lib.query("sbgm_conv2d_tc_workspace_bytes", self.fmt, x.n, x.h, x.w,
                                                              cw.cin, cw.cout, cw.kh, cw.kw, stride, pad)
            part = None
            if gn_stats and residual is None and tproj is None and act == ACT_NONE and proj is None:
                chunks = _lib.query("sbgm_conv2d_tc_gn_chunks", self.fmt, x.n, x.h, x.w, cw.cin, cw.cout, cw.kh, cw.kw, stride, pad)
                if chunks > 0:
                    part = torch.empty((x.n, chunks, cw.cout // 8, 2), dtype=torch.float32, device=self.device)
                    stats = (part, chunks)
            ws = None
            if ws_bytes:
                if self._splitk_ws is None or self._splitk_ws.numel() * 4 < ws_bytes:
                    self._splitk_ws = torch.empty(ws_bytes // 4, dtype=torch.float32, device=self.device)
                ws = self._splitk_ws.data_ptr()
            call("sbgm_conv2d_tc", x.ptr, x.plane, cw.w.data_ptr(), cw.plane, _ptr(cw.bias), res_ptr, res_plane,
                 tp_ptr, tp_stride, out_ptr, out_plane, self.fmt, x.n, x.h, x.w, cw.cin, cw.cout, cw.kh, cw.kw,
                 stride, pad, act, *pargs, ws, ws_bytes, _ptr(part), _stream())
        if proj is not None:
            return (out, pout) if proj_keep else pout
        return (out, stats) if gn_stats else out

    def stem_im2col(self, x: torch.Tensor, planes: Optional[torch.Tensor], c_begin: int, c_end: int, cc: int) -> Act:
        """8x8 stride-2 window of channels [c_begin, c_end) of x || planes as an NHWC tensor with 64 channels per input channel."""
        n, _, h, w = x.shape
        out = Act(self.fmt, n, h // 2, w // 2, (c_end - c_begin) * 64, self.device)
        call("sbgm_stem_im2col", x.data_ptr(), _ptr(planes), 1 if planes is None else planes.shape[0], cc, c_begin, c_end,
             out.ptr, out.plane, self.fmt, n, h, w, _stream())
        return out

    def linear(self, x: Act, cw: ConvW, act: int = ACT_NONE, residual: Optional[Act] = None) -> Act:
        return self.conv(x, cw, 1, 0, act, residual)

    def linear_ln(self, x: Act, cw: ConvW, act: int = ACT_NONE) -> Act:
        """act(LayerNorm(x) W^T + b) with the LayerNorm folded into the GEMM (`cw` from pack_linear_ln)."""
        rows = x.n * x.h * x.w
        out = Act(self.fmt, 1, 1, rows, cw.cout, self.device)
        if "conv_tc" in _SKIP or "tc_1x1" in _SKIP:
            return out
        call("sbgm_linear_ln_tc", x.ptr, x.plane, cw.w.data_ptr(), cw.plane, cw.bias.data_ptr(), cw.colsum.data_ptr(), LN_EPS, out.ptr,
             out.plane, self.fmt, rows, cw.cin, cw.cout, act, _stream())
        return out

    def groupnorm(self, x: Act, gamma, beta, groups: int, act: int = ACT_NONE, skip: Optional[Act] = None,
                  tproj: Optional[torch.Tensor] = None, stats=None) -> Act:
        if "gn" in _SKIP:
            return x
        if stats is not None and (x.c // 8) % groups == 0:
            part, chunks = stats
            out = x.like()
            call("sbgm_groupnorm_apply", x.ptr, x.plane, part.data_ptr(), chunks, x.c // 8, _ptr(gamma), _ptr(beta), groups, GN_EPS,
                 None if skip is None else skip.ptr, 0 if skip is None else skip.plane,
                 _ptr(tproj), tproj.stride(0) if tproj is not None else 0, act, out.ptr, out.plane, self.fmt,
                 x.n, x.h * x.w, x.c, _stream())
            return out
        need = _lib.query("sbgm_groupnorm_scratch_floats", x.n, x.c, x.h * x.w)
        if self._gn_scratch is None or self._gn_scratch.numel() < need:
            self._gn_scratch = torch.empty(need, dtype=torch.float32, device=self.device)
        out = x.like()
        call("sbgm_groupnorm", x.ptr, x.plane, _ptr(gamma), _ptr(beta), groups, GN_EPS,
             None if skip is None else skip.ptr, 0 if skip is None else skip.plane,
             _ptr(tproj), tproj.stride(0) if tproj is not None else 0, act, out.ptr, out.plane, self.fmt,
             x.n, x.h * x.w, x.c, self._gn_scratch.data_ptr(), _stream())
        return out

    def up_fused_ok(self, x: Act, cw: ConvW) -> bool:
        """True if conv3x3(upsample2x(x)) runs as ONE kernel (sbgm_conv3x3_c64_up): a 64 -> 64 convolution in a single-plane format."""
        return (self.fmt in (FMT_BF16, FMT_F16) and x.c == 64 and cw.cin == 64 and cw.cout == 64 and cw.kh == 3
                and cw.kw == 3 and (2 * x.h) % 16 == 0 and (2 * x.w) % 8 == 0 and not _SKIP)

    def conv_up_fused(self, x: Act, cw: ConvW, proj: Optional[torch.Tensor] = None, gn_stats: bool = False):
        """conv3x3(upsample2x(x)) with the bilinear resize inside the kernel's operand stage.  Returns like `conv`: the projected
        tensor (`proj`), (Act, stats) (`gn_stats`) or the Act."""
        h, w = 2 * x.h, 2 * x.w
        if CONV_TRACE is not None:
            CONV_TRACE.append(dict(n=x.n, h=h, w=w, cw=cw, stride=1, pad=1, act=ACT_NONE, residual=False, tproj=False,
                                   proj=proj is not None, gn_stats=gn_stats, c64=True, up_fused=True))
        out, pout, part, stats = None, None, None, None
        if proj is not None:
            pout = torch.empty((x.n, h, w, _lib.PROJ_STRIDE), dtype=torch.float32, device=self.device)
            pargs = (proj.data_ptr(), proj.shape[0], pout.data_ptr())
        else:
            out = Act(self.fmt, x.n, h, w, cw.cout, self.device)
            pargs = (None, 0, None)
            if gn_stats:
                chunks = (h // 16) * (w // 8) * 4
                part = torch.empty((x.n, chunks, 8, 2), dtype=torch.float32, device=self.device)
                stats = (part, chunks)
        call("sbgm_conv3x3_c64_up", x.ptr, x.plane, cw.w.data_ptr(), cw.plane, _ptr(cw.bias), None if out is None else out.ptr,
             0 if out is None else out.plane, self.fmt, x.n, h, w, ACT_NONE, *pargs, _ptr(part), 8, _stream())
        if proj is not None:
            return pout
        return (out, stats) if gn_stats else out

    def affine(self, x: Act, skip: Optional[Act] = None, tproj: Optional[torch.Tensor] = None, act: int = ACT_NONE,
               bias: Optional[torch.Tensor] = None) -> Act:
        """act(x + bias + skip + tproj) as the normalisation kernel with unit statistics (mean 0, rstd 1, no gamma): the epilogue
        of a decoder block whose norm is nn.Identity (score_unet.py:593-612), or the bias of the fp32 transposed convolution.
        The tproj-before-activation flag is inert without a tproj; the bias form passes 0."""
        unit = torch.tensor([0.0, 1.0], dtype=torch.float32, device=self.device).repeat(x.c, 1).contiguous()
        out = x.like()
        call("sbgm_norm_apply", x.ptr, x.plane, unit.data_ptr(), 2, x.c, None, _ptr(bias), None if skip is None else skip.ptr,
             0 if skip is None else skip.plane, _ptr(tproj), tproj.stride(0) if tproj is not None else 0, int(bias is None), act,
             out.ptr, out.plane, self.fmt, x.n, x.h * x.w, x.c, _stream())
        return out

    def conv_transpose2x(self, x: Act, tw: TransposeW) -> Act:
        if self.fmt == FMT_F32:
            # the data gradient of a (2x2, stride 2) convolution IS the transposed convolution; the bias is added afterwards
            raw = Act(self.fmt, x.n, 2 * x.h, 2 * x.w, tw.cout, self.device)
            call("sbgm_conv2d_dgrad_simt", x.ptr, x.plane, tw.simt.data_ptr(), raw.ptr, raw.plane, 0, self.fmt,
                 x.n, 2 * x.h, 2 * x.w, tw.cout, tw.cin, 2, 2, 2, 0, _stream())
            return self.affine(raw, bias=tw.bias)
        out = Act(self.fmt, x.n, 2 * x.h, 2 * x.w, tw.cout, self.device)
        for a, b, cw in tw.subs:
            call("sbgm_conv2d_tc_ex", x.ptr, x.plane, cw.w.data_ptr(), cw.plane, cw.bias.data_ptr(), None, 0, 0, None, 0, out.ptr, out.plane,
                 self.fmt, x.n, x.h, x.w, cw.cin, cw.cout, 1, 1, 1, 0, 0, x.h, x.w, 2 * x.h, 2 * x.w, 2, a, b, ACT_NONE, None, 0, _stream())
        return out

    def final_conv(self, a: Act, w: torch.Tensor, bias: torch.Tensor, inv_std: InvStd, out: torch.Tensor) -> None:
        """out [n, cout, h, w] fp32 = (conv3x3(a, w) + bias) * 1/std: the decoder's final layer (`w` [cout][9][cin] fp32)."""
        call("sbgm_final_conv", a.ptr, a.plane, self.fmt, w.data_ptr(), bias.data_ptr(), *inv_std.args(), out.data_ptr(),
             a.n, a.h, a.w, a.c, w.shape[0], _stream())

    def final_gather(self, proj: torch.Tensor, bias: torch.Tensor, inv_std: InvStd, out: torch.Tensor) -> None:
        """The final 64 -> 1 layer from the nine per-tap partial products `proj` [n, h, w, PROJ_STRIDE] that conv_up's epilogue
        emitted: out [n, 1, h, w] = (sum of the taps + bias) * 1/std."""
        n, h, w = proj.shape[:3]
        call("sbgm_final_gather", proj.data_ptr(), bias.data_ptr(), *inv_std.args(), out.data_ptr(), n, h, w, _stream())

    def layernorm(self, x: Act, gamma, beta) -> Act:
        if "ln" in _SKIP:
            return x
        out = x.like()
        rows = x.n * x.h * x.w
        call("sbgm_layernorm", x.ptr, x.plane, gamma.data_ptr(), beta.data_ptr(), LN_EPS, out.ptr, out.plane, self.fmt,
             rows, x.c, _stream())
        return out

    def upsample2x(self, x: Act) -> Act:
        out = x.like(h=2 * x.h, w=2 * x.w)
        if "upsample" in _SKIP:
            return out
        call("sbgm_upsample2x", x.ptr, x.plane, out.ptr, out.plane, self.fmt, x.n, x.h, x.w, x.c, _stream())
        return out

    def attention_out_proj_ok(self, b: int, s: int, c: int, heads: int) -> bool:
        """True if the attention core + out-projection + residual run as one tcgen05 kernel (csrc/attn_fused.cu): where the
        kernel supports the shape and it measured faster than the two launches it replaces, i.e. with enough query tiles to fill
        the GPU (16 x 16 maps at the benchmark batch)."""
        if "attn_core" in _SKIP or not _lib.query("sbgm_attention_out_proj_supported", self.fmt, b, s, c, heads):
            return False
        return b * s >= 128 * 96

    def attention_out_proj(self, qkv: Act, x: Act, cw: ConvW, b: int, s: int, c: int, heads: int) -> Act:
        """x + out_proj(softmax(Q K^T / sqrt(d)) V): scores, probabilities and head outputs stay on the SM."""
        out = Act(self.fmt, 1, 1, b * s, c, self.device)
        call("sbgm_attention_out_proj", qkv.ptr, x.ptr, cw.w.data_ptr(), cw.plane, cw.bias.data_ptr(), out.ptr, self.fmt, b, s, c, heads,
             _stream())
        return out

    def attention_core(self, qkv: Act, b: int, s: int, c: int, heads: int) -> Act:
        out = Act(self.fmt, 1, 1, b * s, c, self.device)
        if "attn_core" in _SKIP:
            return out
        call("sbgm_attention", qkv.ptr, qkv.plane, out.ptr, out.plane, self.fmt, b, s, c, heads, _stream())
        return out


class AttentionW:
    def __init__(self, pk: _Packer, keys: "AttnKeys", heads: int) -> None:
        self.heads = heads
        self.ln1 = (pk.vec(keys.ln1.weight), pk.vec(keys.ln1.bias))
        self.ln2 = (pk.vec(keys.ln2.weight), pk.vec(keys.ln2.bias))
        self.in_proj = pk.conv(*keys.in_proj)
        self.out_proj = pk.conv(*keys.out_proj)
        self.ff0 = pk.conv(*keys.ff0)
        self.ff2 = pk.conv(*keys.ff2)
        # LayerNorm folded into the Linear layer behind it (tensor-core formats): ln1 -> in_proj, ln2 -> ff.0
        self.fold = pk.fmt != FMT_F32
        if self.fold:
            self.in_proj_ln = pack_linear_ln(pk, *keys.in_proj, *keys.ln1)
            self.ff0_ln = pack_linear_ln(pk, *keys.ff0, *keys.ln2)


def attention_block(k: Kernels, aw: AttentionW, x: Act) -> Act:
    """ImageSelfAttention.forward (score_unet.py:136-148) on NHWC tokens (the flatten is free)."""
    if "attn" in _SKIP:
        return x
    tok = x.tokens()
    b, s, c = x.n, x.h * x.w, x.c
    fold = aw.fold and "ln" not in _SKIP
    qkv = k.linear_ln(tok, aw.in_proj_ln) if fold else k.linear(k.layernorm(tok, *aw.ln1), aw.in_proj)
    if k.attention_out_proj_ok(b, s, c, aw.heads):
        h = k.attention_out_proj(qkv, tok, aw.out_proj, b, s, c, aw.heads)
    else:
        att = k.attention_core(qkv, b, s, c, aw.heads)
        h = k.linear(att, aw.out_proj, residual=tok)
    g = k.linear_ln(h, aw.ff0_ln, act=ACT_GELU) if fold else k.linear(k.layernorm(h, *aw.ln2), aw.ff0, act=ACT_GELU)
    return k.linear(g, aw.ff2, residual=h).view(x.n, x.h, x.w, x.c)


class TimeProjector:
    """All Gaussian-Fourier embeddings and SiLU->Linear projections in one launch.

    Heads are addressed by name; `cols(name)` gives the column slice of the [rows, c_total] output.
    """

    def __init__(self, device, te: int) -> None:
        self.device, self.te = device, te
        self.sets: List[torch.Tensor] = []
        self.w: List[torch.Tensor] = []
        self.b: List[torch.Tensor] = []
        self.set_of: List[torch.Tensor] = []
        self.slices: Dict[str, Tuple[int, int]] = {}
        self.label_emb: Optional[torch.Tensor] = None
        self.c_total = 0
        self._packed = None

    def add_set(self, W: torch.Tensor) -> int:
        self.sets.append(W.reshape(-1))
        return len(self.sets) - 1

    def add_head(self, name: str, set_idx: int, w: torch.Tensor, b: torch.Tensor) -> None:
        c = w.shape[0]
        self.slices[name] = (self.c_total, self.c_total + c)
        self.c_total += c
        self.w.append(w)
        self.b.append(b)
        self.set_of.append(torch.full((c,), set_idx, dtype=torch.int32, device=self.device))

    def add_heads(self, heads: Sequence["TimeHead"], get: Callable[[str], torch.Tensor]) -> None:
        """Add the layout's heads in column order; heads naming the same Fourier W share one set.  `get(key)`: a key's tensor."""
        sets: Dict[str, int] = {}
        for h in heads:
            if h.fourier not in sets:
                sets[h.fourier] = self.add_set(get(h.fourier))
            self.add_head(h.name, sets[h.fourier], get(h.weight), get(h.bias))

    def finalize(self) -> None:
        self._packed = (torch.stack(self.sets).contiguous(), torch.cat(self.w).contiguous(),
                        torch.cat(self.b).contiguous(), torch.cat(self.set_of).contiguous())

    def __call__(self, t: torch.Tensor, y: Optional[torch.Tensor], *, rows: Optional[int] = None,
                 t_row_stride: int = 1, t_step_stride: int = 0, step_counter: Optional[torch.Tensor] = None,
                 out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Projection table [rows, c_total].  Default: one row per element of `t`.  A sampler passes its
        step table as `t` with t_row_stride=0, t_step_stride=STEP_COLS and the device step counter."""
        fw, pw, pb, ps = self._packed
        if rows is None:
            rows = t.numel()
            t = t.reshape(-1).to(device=self.device, dtype=torch.float32).contiguous()
        yy = None if y is None else y.reshape(-1).to(device=self.device, dtype=torch.int64).contiguous()
        if yy is not None and yy.numel() != rows:
            raise ValueError(f"Batch mismatch: x= {rows}, y={yy.numel()}.")
        if out is None:
            out = torch.empty((rows, self.c_total), dtype=torch.float32, device=self.device)
        call("sbgm_time_embed_project", t.data_ptr(), t_row_stride, t_step_stride, _ptr(step_counter), _ptr(yy),
             fw.data_ptr(), fw.shape[0], self.te, _ptr(self.label_emb) if yy is not None else None, pw.data_ptr(),
             pb.data_ptr(), ps.data_ptr(), self.c_total, out.data_ptr(), rows, _stream())
        return out

    def cols(self, table: torch.Tensor, name: str) -> torch.Tensor:
        a, b = self.slices[name]
        return table[:, a:b]


# -- checkpoint layout ----------------------------------------------------------------------------------------------------
# The state-dict keys of the score-UNet (the reference's checkpoint format, mirrored by score_unet.py's module tree), as plain
# records in forward order, under a key prefix: "" for a standalone module's own state dict.  Both engines read the network
# through them, and keep their packed weights in records of the same types, under the same field names.
Affine = namedtuple("Affine", "weight bias")                              # a convolution, Linear or normalisation layer
BatchNormKeys = namedtuple("BatchNormKeys", "weight bias running_mean running_var")
ConvBN = namedtuple("ConvBN", "conv bn")                                  # a convolution without bias + the BatchNorm2d behind it
AttnKeys = namedtuple("AttnKeys", "ln1 in_proj out_proj ln2 ff0 ff2")     # ImageSelfAttention, in forward order
# one SiLU -> Linear time projection: its TimeProjector head name, the key of its Fourier features' W, its Linear
TimeHead = namedtuple("TimeHead", "name fourier weight bias")
# a BasicBlock: ConvBN sites (down: the 1x1 downsample or None) and the stride of conv1 and the downsample
EncBlock = namedtuple("EncBlock", "c1 c2 down stride")
# stem: conv1.weight; attn: {stage: the AttnKeys behind it}; heads: enc0 (the stem) .. enc4 (stage 4), sharing one Fourier W
EncoderLayout = namedtuple("EncoderLayout", "stem conv2 stages attn heads label_emb")
# a DecoderBlock: conv_up is the resize convolution or the transposed convolution; n1 / n2: the GroupNorm's Affine, None for
# InstanceNorm or nn.Identity; g1 / g2: the group counts (the channel count for InstanceNorm); head: its TimeHead
DecBlock = namedtuple("DecBlock", "conv_up conv n1 n2 g1 g2 attn head")
DecoderLayout = namedtuple("DecoderLayout", "blocks final_up final_conv")   # final_up: final_layer's up-path, as DecBlock.conv_up


def _affine(p: str) -> Affine:
    return Affine(f"{p}weight", f"{p}bias")


def batchnorm_keys(p: str) -> BatchNormKeys:
    return BatchNormKeys(f"{p}.weight", f"{p}.bias", f"{p}.running_mean", f"{p}.running_var")


def attention_layout(p: str) -> AttnKeys:
    return AttnKeys(_affine(f"{p}ln1."), Affine(f"{p}mha.in_proj_weight", f"{p}mha.in_proj_bias"), _affine(f"{p}mha.out_proj."),
                    _affine(f"{p}ln2."), _affine(f"{p}ff.0."), _affine(f"{p}ff.2."))


def encoder_layout(spec: "UNetSpec", p: str = "encoder.") -> EncoderLayout:
    conv_bn = lambda conv, bn: ConvBN(f"{conv}weight", batchnorm_keys(bn))
    stages, inplanes = [], FMAP_CHANNELS[0]
    for li, nblk in enumerate(spec.block_layers, start=1):
        planes, blocks = FMAP_CHANNELS[li], []
        for b in range(nblk):
            bp = f"{p}layer{li}.{b}."
            stride = 2 if (b == 0 and li > 1) else 1
            down = conv_bn(f"{bp}downsample.0.", f"{bp}downsample.1") if stride != 1 or inplanes != planes else None
            blocks.append(EncBlock(conv_bn(f"{bp}conv1.", f"{bp}bn1"), conv_bn(f"{bp}conv2.", f"{bp}bn2"), down, stride))
            inplanes = planes
        stages.append(tuple(blocks))
    heads = tuple(TimeHead(f"enc{i}", f"{p}sinusoidal_embedding.W", f"{p}time_projection_layers.{i}.1.weight",
                           f"{p}time_projection_layers.{i}.1.bias") for i in range(len(FMAP_CHANNELS)))
    return EncoderLayout(f"{p}conv1.weight", conv_bn(f"{p}conv2.", f"{p}bn1"), tuple(stages),
                         {i: attention_layout(f"{p}attention_layers.{i}.") for i in (3, 4)}, heads,
                         f"{p}label_emb.weight" if spec.has_labels else None)


def _up_site(p: str, use_resize_conv: bool) -> Affine:
    return _affine(f"{p}conv_up." if use_resize_conv else f"{p}transpose.")


def decoder_block_layout(p: str, head: str, cin: int, cout: int, attn: bool, norm: str, gn_groups: int,
                         use_resize_conv: bool) -> DecBlock:
    group = norm == "group"
    return DecBlock(_up_site(p, use_resize_conv), _affine(f"{p}conv."), _affine(f"{p}norm1.") if group else None,
                    _affine(f"{p}norm2.") if group else None, max(1, min(gn_groups, cin)) if group else cin,
                    max(1, min(gn_groups, cout)) if group else cout, attention_layout(f"{p}attention.") if attn else None,
                    TimeHead(head, f"{p}sinusoidal_embedding.W", f"{p}time_projection_layer.1.weight", f"{p}time_projection_layer.1.bias"))


def decoder_layout(spec: "UNetSpec", p: str = "decoder.") -> DecoderLayout:
    """The final layer runs without a time input: its Fourier W and time projection are not part of the layout."""
    blocks = tuple(decoder_block_layout(f"{p}residual_layers.{i}.", f"dec{i}", cin, cout, attn, spec.norm, spec.gn_groups,
                                        spec.use_resize_conv) for i, (cin, cout, attn) in enumerate(spec.plan))
    return DecoderLayout(blocks, _up_site(f"{p}final_layer.", spec.use_resize_conv), _affine(f"{p}final_layer.conv."))


def stem_matrix(w1: torch.Tensor) -> torch.Tensor:              # conv1.weight [64][cin][8][8] -> the stem kernels' [cin][tap][co]
    return w1.permute(1, 2, 3, 0).reshape(w1.shape[1], 64, 64).contiguous()


def final_matrix(wf: torch.Tensor) -> torch.Tensor:             # final_layer.conv.weight [cout][cin][3][3] -> [cout][tap][cin]
    return wf.permute(0, 2, 3, 1).reshape(wf.shape[0], 9, wf.shape[1]).contiguous()


class EncoderEngine:
    def __init__(self, sd, spec: "UNetSpec", lay: EncoderLayout, *, fmt: int, device, tp: TimeProjector) -> None:
        pk = _Packer(sd, fmt, device)
        self.k = Kernels(fmt, device)
        self.fmt, self.device, self.tp = fmt, device, tp
        w1 = pk.get(lay.stem)                                            # [64, cin, 8, 8]
        self.cin = w1.shape[1]
        self.stem_w = stem_matrix(w1)
        if fmt != FMT_F32:
            # tensor-core stem: conv1 as a 1x1 convolution over the im2col tensor (K index = ci * 64 + r * 8 + s = OIHW order)
            km = lambda wsub: pack_tc_matrix(wsub.reshape(64, -1).contiguous(), fmt)
            self.stem_cw_all = ConvW(km(w1), None, self.cin * 64, 64, 1, 1)
            self.stem_cw_x = ConvW(km(w1[:, :1]), None, 64, 64, 1, 1)
        conv_bn = lambda s: pk.conv(s.conv, bn=s.bn)
        self.conv2 = conv_bn(lay.conv2)
        self.layers = [[s._replace(down=None if s.down is None else conv_bn(s.down), c1=conv_bn(s.c1), c2=conv_bn(s.c2))
                        for s in stage] for stage in lay.stages]
        self.attn = {i: AttentionW(pk, keys, spec.n_heads) for i, keys in lay.attn.items()}
        tp.add_heads(lay.heads, pk.get)
        if lay.label_emb is not None:
            tp.label_emb = pk.get(lay.label_emb).contiguous()

    def alloc_partial(self, npl: int, h: int, w: int):
        """Buffer for `stem_partial`: fp32 NHWC tensor (fp32 mode) or an `Act` in the engine's format (tensor-core modes,
        where it enters the stem convolution's epilogue as a residual)."""
        if self.fmt == FMT_F32:
            return torch.empty((npl, h // 2, w // 2, 64), dtype=torch.float32, device=self.device)
        return Act(self.fmt, npl, h // 2, w // 2, 64, self.device)

    def stem_partial(self, planes: torch.Tensor, h: int, w: int, out=None):
        """conv1 restricted to the conditioning channels (step-invariant in a sampler)."""
        npl, cc = planes.shape[0], planes.shape[1]
        if out is None:
            out = self.alloc_partial(npl, h, w)
        f32 = out if self.fmt == FMT_F32 else torch.empty((npl, h // 2, w // 2, 64), dtype=torch.float32, device=self.device)
        assert tuple(f32.shape) == (npl, h // 2, w // 2, 64) and f32.is_contiguous()
        call("sbgm_stem_conv", None, planes.data_ptr(), npl, cc, 1, cc + 1, self.stem_w.data_ptr(), None, 0, None, 0,
             f32.data_ptr(), f32.numel(), FMT_F32, npl, h, w, _stream())
        if self.fmt != FMT_F32:
            assert (out.n, out.h, out.w, out.c) == (npl, h // 2, w // 2, 64)
            call("sbgm_convert", f32.data_ptr(), 0, FMT_F32, out.ptr, out.plane, self.fmt, f32.numel(), _stream())
        return out

    def forward(self, x: torch.Tensor, planes: Optional[torch.Tensor], tproj: torch.Tensor,
                partial: Optional[torch.Tensor] = None) -> List[Act]:
        """x [n,1,h,w] fp32; planes [n or 1, cin-1, h, w] fp32 (conditioning channels in concat order)
        or, when `partial` is given, their precomputed stem contribution."""
        k, tp = self.k, self.tp
        n, _, h, w = x.shape
        cc = self.cin - 1
        t0 = tp.cols(tproj, "enc0")
        if self.fmt != FMT_F32:
            # conv1 on the tensor cores: im2col of the 8x8 stride-2 window, then a 1x1 implicit GEMM (K = 64 per channel)
            if (partial is not None or cc == 0) and h % 16 == 0 and w % 32 == 0:
                # one kernel: windows of x built in shared memory, MMA against the resident 64 x 64 weights, + partial + time
                f1 = Act(self.fmt, n, h // 2, w // 2, 64, self.device)
                call("sbgm_stem_x_tc", x.data_ptr(), self.stem_cw_x.w.data_ptr(), self.stem_cw_x.plane,
                     None if partial is None else partial.ptr, 0 if partial is None else partial.plane, 0 if partial is None else partial.n,
                     t0.data_ptr(), t0.stride(0), f1.ptr, f1.plane, self.fmt, n, h, w, _stream())
            else:
                assert partial is None, f"a precomputed stem partial needs h % 16 == 0 and w % 32 == 0, got {h} x {w}"
                if cc > 0:
                    assert planes is not None and planes.shape[1] == cc, f"encoder expects {cc} conditioning channels"
                f1 = k.conv(k.stem_im2col(x, planes, 0, self.cin, cc), self.stem_cw_all, tproj=t0)
            return self._after_stem(f1, tproj)
        f1 = Act(self.fmt, n, h // 2, w // 2, 64, self.device)
        if partial is not None:
            call("sbgm_stem_conv", x.data_ptr(), None, 1, cc, 0, 1, self.stem_w.data_ptr(), partial.data_ptr(),
                 partial.shape[0], t0.data_ptr(), t0.stride(0), f1.ptr, f1.plane, self.fmt, n, h, w, _stream())
        else:
            if cc > 0:
                assert planes is not None and planes.shape[1] == cc, f"encoder expects {cc} conditioning channels"
            call("sbgm_stem_conv", x.data_ptr(), _ptr(planes), 1 if planes is None else planes.shape[0], cc, 0, self.cin,
                 self.stem_w.data_ptr(), None, 0, t0.data_ptr(), t0.stride(0), f1.ptr, f1.plane, self.fmt, n, h, w, _stream())
        return self._after_stem(f1, tproj)

    def _after_stem(self, f1: Act, tproj: torch.Tensor) -> List[Act]:
        k, tp = self.k, self.tp
        fmaps = [f1]
        hcur = k.conv(f1, self.conv2, stride=2, pad=3, act=ACT_RELU)
        for li, blocks in enumerate(self.layers, start=1):
            for bi, (c1, c2, down, stride) in enumerate(blocks):
                last = bi == len(blocks) - 1
                idn = hcur if down is None else k.conv(hcur, down, stride=stride, pad=0)
                mid = k.conv(hcur, c1, stride=stride, pad=1, act=ACT_RELU)
                hcur = k.conv(mid, c2, stride=1, pad=1, act=ACT_RELU, residual=idn,
                              tproj=tp.cols(tproj, f"enc{li}") if last else None)
            if li in self.attn:
                hcur = attention_block(k, self.attn[li], hcur)
            fmaps.append(hcur)
        return fmaps


def pack_decoder_block(pk: _Packer, s: DecBlock, use_resize_conv: bool, n_heads: int) -> DecBlock:
    norm = lambda a: (None, None) if a is None else (pk.vec(a.weight), pk.vec(a.bias))      # n1 / n2: (gamma, beta)
    return s._replace(conv_up=pk.up(s.conv_up, use_resize_conv), conv=pk.conv(*s.conv), n1=norm(s.n1), n2=norm(s.n2),
                      attn=None if s.attn is None else AttentionW(pk, s.attn, n_heads))


class DecoderEngine:
    def __init__(self, sd, spec: "UNetSpec", lay: DecoderLayout, *, fmt: int, device, tp: TimeProjector) -> None:
        pk = _Packer(sd, fmt, device)
        self.k = Kernels(fmt, device)
        self.fmt, self.device, self.tp = fmt, device, tp
        self.use_resize_conv, self.out_channels, self.act = spec.use_resize_conv, spec.out_channels, ACTS[spec.activation]
        self.blocks = [pack_decoder_block(pk, s, spec.use_resize_conv, spec.n_heads) for s in lay.blocks]
        tp.add_heads([s.head for s in lay.blocks], pk.get)
        self.final_up = pk.up(lay.final_up, spec.use_resize_conv)
        self.final_w = final_matrix(pk.get(lay.final_conv.weight))
        self.final_b = pk.vec(lay.final_conv.bias)

    def forward(self, fmaps: List[Act], tproj: torch.Tensor, inv_std: InvStd, dst: Optional[torch.Tensor] = None) -> torch.Tensor:
        k, tp = self.k, self.tp
        rev = list(reversed(fmaps))
        out = rev[0]
        for i, blk in enumerate(self.blocks):
            if self.use_resize_conv and k.up_fused_ok(out, blk.conv_up):
                a, st1 = k.conv_up_fused(out, blk.conv_up, gn_stats=True)       # the bilinear upsample inside the operand stage
            elif self.use_resize_conv:
                up = k.upsample2x(out)
                a, st1 = k.conv(up, blk.conv_up, pad=1, gn_stats=True)
            else:
                a, st1 = k.conv_transpose2x(out, blk.conv_up), None
            a = k.groupnorm(a, *blk.n1, groups=blk.g1, stats=st1)
            b, st2 = k.conv(a, blk.conv, pad=1, gn_stats=True)
            skip = rev[i + 1]
            if (skip.n, skip.h, skip.w, skip.c) != (b.n, b.h, b.w, b.c):
                raise AssertionError(f"prev_fmap shape {(skip.n, skip.c, skip.h, skip.w)} must match output shape {(b.n, b.c, b.h, b.w)}")
            out = k.groupnorm(b, *blk.n2, groups=blk.g2, act=self.act, skip=skip, tproj=tp.cols(tproj, blk.head.name), stats=st2)
            if blk.attn is not None:
                out = attention_block(k, blk.attn, out)
        # the final layer: conv_up's output `a` for the final convolution, or the final 64 -> 1 convolution's per-tap partial
        # products `pr` out of conv_up's epilogue (its 64-channel output never reaches HBM; tc_common.cuh: projection epilogue)
        a = pr = None
        if self.use_resize_conv and k.up_fused_ok(out, self.final_up):
            if self.out_channels == 1:
                pr = k.conv_up_fused(out, self.final_up, proj=self.final_w[0])
            else:
                a = k.conv_up_fused(out, self.final_up)
        elif not self.use_resize_conv:
            a = k.conv_transpose2x(out, self.final_up)
        elif self.fmt != FMT_F32 and self.out_channels == 1 and self.final_up.cout == 64:
            pr = k.conv(k.upsample2x(out), self.final_up, pad=1, proj=self.final_w[0])
        else:
            a = k.conv(k.upsample2x(out), self.final_up, pad=1)
        n, h, w = (a.n, a.h, a.w) if pr is None else pr.shape[:3]
        res = dst if dst is not None else torch.empty((n, self.out_channels, h, w), dtype=torch.float32, device=self.device)
        if pr is None:
            k.final_conv(a, self.final_w, self.final_b, inv_std, res)
        else:
            k.final_gather(pr, self.final_b, inv_std, res)
        return res


def concat_planes(x_batch: int, lsm, topo, cond, device) -> Optional[torch.Tensor]:
    """Conditioning channels in the reference's concat order lsm || topo || cond_img (score_unet.py:273-291)."""
    parts = []
    for name, c in (("lsm_cond", lsm), ("topo_cond", topo), ("cond_img", cond)):
        if c is None:
            continue
        if name != "cond_img" and c.shape[0] != x_batch:
            raise ValueError(f"Batch mismatch: x= {x_batch}, {name}={c.shape[0]}.")
        parts.append(c.to(device=device, dtype=torch.float32))
    if not parts:
        return None
    return torch.cat(parts, dim=1).contiguous()


@dataclass
class UNetSpec:
    """Architecture knobs recovered from the module tree (they mirror the reference constructors)."""
    time_embedding: int = 256
    block_layers: Tuple[int, ...] = (2, 2, 2, 2)
    n_heads: int = 4
    has_labels: bool = False
    plan: Tuple[Tuple[int, int, bool], ...] = ((512, 256, True), (256, 128, True), (128, 64, False), (64, 64, False))
    out_channels: int = 1
    use_resize_conv: bool = True
    norm: str = "group"
    gn_groups: int = 8
    activation: str = "silu"


def engine_device(precision: str, device) -> torch.device:
    """Check an engine's precision name and device and load the library; returns the device."""
    if precision not in PRECISIONS:
        raise ValueError(f"precision must be one of {sorted(PRECISIONS)}, got {precision!r}")
    device = torch.device(device)
    if device.type != "cuda":
        raise RuntimeError("sbgm_danra_b200 runs on CUDA devices only (no CPU fallback); got device " + str(device))
    _lib.load_library()
    return device


class UNetEngine:
    """Encoder + decoder + time projector packed for one (state-dict, precision, device)."""

    def __init__(self, sd: Dict[str, torch.Tensor], spec: UNetSpec, precision: str, device) -> None:
        device = engine_device(precision, device)
        self.spec, self.precision, self.device = spec, precision, device
        self.fmt = PRECISIONS[precision]
        with torch.cuda.device(device), torch.no_grad():
            self.tp = TimeProjector(device, spec.time_embedding)
            self.enc = EncoderEngine(sd, spec, encoder_layout(spec), fmt=self.fmt, device=device, tp=self.tp)
            self.dec = DecoderEngine(sd, spec, decoder_layout(spec), fmt=self.fmt, device=device, tp=self.tp)
            self.tp.finalize()

    def check_input(self, x: torch.Tensor) -> None:
        if x.dim() != 4 or x.shape[1] != 1:
            raise ValueError(f"x must be [B, 1, H, W], got {tuple(x.shape)}")
        if x.shape[2] % 32 != 0 or x.shape[3] % 32 != 0:
            raise ValueError(f"H and W must be multiples of 32 (five stride-2 stages), got {tuple(x.shape[2:])}")

    def forward(self, x: torch.Tensor, t: torch.Tensor, y=None, planes: Optional[torch.Tensor] = None,
                inv_std: Optional[torch.Tensor] = None) -> torch.Tensor:
        """One UNet evaluation: out[n,co,h,w] = decoder(encoder(x, planes, t, y)) * inv_std[n]."""
        self.check_input(x)
        with torch.cuda.device(self.device):
            x = x.to(device=self.device, dtype=torch.float32).contiguous()
            tproj = self.tp(t, y)
            fmaps = self.enc.forward(x, planes, tproj)
            return self.dec.forward(fmaps, tproj, InvStd(inv_std))
