"""Training-mode execution of the score-UNet: forward with batch statistics + a reverse tape of CUDA kernels.

The reference trains through torch autograd (sbgm/training.py:323-410 calls `loss_fn` -> `loss.backward()`,
sbgm/score_unet.py:936-985).  Here one `torch.autograd.Function` (score_unet._ScoreNetFn) wraps the whole
network: its forward runs `TrainEngine.forward`, which sequences the same forward kernels as inference but
with unfolded BatchNorm (batch statistics, running-stat update) and records, per kernel, a closure that
launches the matching backward kernels of `include/sbgm_b200.h` (convolution data / weight gradients on the
tensor cores, normalisation / attention / upsample / time-embedding backward).  `TrainEngine.backward`
replays the closures in reverse and returns fp32 gradients in torch's parameter layouts, written as views of
ONE flat buffer so that data-parallel training can all-reduce it in place (parallel.py).

torch supplies memory, streams and the autograd hook; every FLOP runs in this repo's kernels.
"""
from __future__ import annotations

import ctypes
from typing import Callable, Dict, List, Optional, Sequence, Tuple

import torch

from . import _lib
from ._capture import graph_capture
from ._lib import ACT_GELU, ACT_NONE, ACT_RELU, FMT_BF16X2, FMT_F32, call
from .engine import (ACTS, BN_EPS, GN_EPS, LN_EPS, PRECISIONS, Act, Affine, AttnKeys, ConvBN, ConvW, DecBlock, InvStd, Kernels,
                     TimeProjector, UNetSpec, _ptr, _stream, decoder_layout, encoder_layout, engine_device, final_matrix,
                     pack_transpose, stem_matrix)

BN_MOMENTUM = 0.1
# keys of the input gradients in the dict TrainEngine.backward returns (next to the parameter names)
DX, DPLANES = "input:x", "input:planes"
# "fp16x2" is an inference storage format (engine.py); a model set to it trains on the bf16x3 kernels
TRAIN_PRECISIONS = dict(PRECISIONS, fp16x2=FMT_BF16X2)


def _pack_oihw(w: torch.Tensor, fmt: int) -> torch.Tensor:
    """OIHW fp32 -> the forward kernels' packed layout (engine._Packer.conv without BatchNorm folding)."""
    cout, cin, kh, kw = w.shape
    if fmt == FMT_F32:
        return w.permute(2, 3, 1, 0).reshape(kh * kw * cin, cout).contiguous()
    return _pack_tc(w, fmt, list(range(kh * kw)), False)


def _pack_tc(w: torch.Tensor, fmt: int, taps: Sequence[int], transpose: bool) -> torch.Tensor:
    """One-launch pack (sbgm_pack_weight): out[o][t][i] = w[co][ci][taps[t]], (o, i) = (ci, co) if transpose."""
    cout, cin, kh, kw = w.shape
    w = w.contiguous()
    oo, ii = (cin, cout) if transpose else (cout, cin)
    planes = 2 if fmt == FMT_BF16X2 else 1
    out = torch.empty((planes, oo, len(taps) * ii), dtype=torch.bfloat16, device=w.device)
    arr = (ctypes.c_int * len(taps))(*taps)
    call("sbgm_pack_weight", w.data_ptr(), cout, cin, kh * kw, arr, len(taps), int(transpose), out.data_ptr(), oo * len(taps) * ii,
         fmt, _stream())
    return out if planes == 2 else out[0]


class _PackJob(ctypes.Structure):        # mirrors sbgm_pack_job (include/sbgm_b200.h)
    _fields_ = [("w", ctypes.c_void_p), ("out", ctypes.c_void_p), ("out_plane", ctypes.c_size_t), ("cout", ctypes.c_int),
                ("cin", ctypes.c_int), ("khw", ctypes.c_int), ("ntaps", ctypes.c_int), ("transpose", ctypes.c_int),
                ("taps", ctypes.c_int * 16)]


class PackPlan:
    """Collects every weight pack of a training step and runs them as one batched launch (sbgm_pack_weights); jobs with more
    than 16 taps (the 8x8 convolution's forward pack) go through the single-weight entry point."""

    def __init__(self, fmt: int) -> None:
        self.fmt = fmt
        self.jobs: List[Tuple[torch.Tensor, torch.Tensor, int, int, int, List[int], bool]] = []

    def add(self, w4: torch.Tensor, taps: Sequence[int], transpose: bool, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """`out`: [planes][o][taps * i] bf16 destination (a slice of a larger table), else a new tensor."""
        cout, cin, kh, kw = w4.shape
        w4 = w4.contiguous()
        oo, ii = (cin, cout) if transpose else (cout, cin)
        planes = 2 if self.fmt == FMT_BF16X2 else 1
        if out is None:
            out = torch.empty((planes, oo, len(taps) * ii), dtype=torch.bfloat16, device=w4.device)
        self.jobs.append((w4, out, cout, cin, kh * kw, list(taps), transpose))
        return out if planes == 2 else out[0]

    def run(self) -> None:
        small = [j for j in self.jobs if len(j[5]) <= 16]
        for w4, out, cout, cin, khw, taps, tr in (j for j in self.jobs if len(j[5]) > 16):
            arr = (ctypes.c_int * len(taps))(*taps)
            call("sbgm_pack_weight", w4.data_ptr(), cout, cin, khw, arr, len(taps), int(tr), out.data_ptr(), out[0].numel(), self.fmt,
                 _stream())
        if small:
            table = (_PackJob * len(small))()
            for k, (w4, out, cout, cin, khw, taps, tr) in enumerate(small):
                e = table[k]
                e.w, e.out, e.out_plane = w4.data_ptr(), out.data_ptr(), out.stride(0)
                e.cout, e.cin, e.khw, e.ntaps, e.transpose = cout, cin, khw, len(taps), int(tr)
                for t, v in enumerate(taps):
                    e.taps[t] = v
            call("sbgm_pack_weights", table, len(small), self.fmt, _stream())
        self.jobs = []


def _dgrad_taps(k: int, stride: int, pad: int, par: int):
    """Taps of a length-k filter that reach input positions of parity `par` in the data gradient, ordered by increasing
    offset d into dy: input index i = stride * j + par receives dy[j + d] * w[r] with r = par + pad - stride * d."""
    ds = sorted(d for d in range(-k, k + 1) if 0 <= par + pad - stride * d < k)
    return ds, [par + pad - stride * d for d in ds]


def stem_dgrad_taps(py: int, px: int) -> List[int]:
    """Flat taps r * 8 + s of Encoder.conv1 (8x8, stride 2, pad 3) that reach input pixels of parity (py, px), in the order of
    sbgm_stem_dgrad_tc's K blocks (increasing offset into df)."""
    return [r * 8 + s for r in _dgrad_taps(8, 2, 3, py)[1] for s in _dgrad_taps(8, 2, 3, px)[1]]


def stem_dgrad_weight(plan: PackPlan, w1: torch.Tensor) -> torch.Tensor:
    """sbgm_stem_dgrad_tc's weight table [4 classes][planes][16][16 * 64]: per parity class (py * 2 + px) conv1.weight, zero-padded
    to 16 input channels, transposed over the class's taps.  Registered on `plan` (filled by plan.run())."""
    w16 = torch.zeros((64, 16, 8, 8), dtype=torch.float32, device=w1.device)
    w16[:, :w1.shape[1]] = w1
    table = torch.empty((4, 2 if plan.fmt == FMT_BF16X2 else 1, 16, 16 * 64), dtype=torch.bfloat16, device=w1.device)
    for cls in range(4):
        plan.add(w16, stem_dgrad_taps(cls >> 1, cls & 1), True, out=table[cls])
    return table


class ConvLayer:
    """One convolution / linear layer of the training graph: forward pack + what its gradients need.

    With a `plan` (and the layer's stride / pad), the forward and data-gradient packs are registered for the batched
    launch instead of being packed one by one."""

    def __init__(self, name: str, w: torch.Tensor, bias: Optional[torch.Tensor], fmt: int, bias_name: Optional[str] = None,
                 plan: Optional[PackPlan] = None, stride: int = 1, pad: int = 0, need_dx: bool = True):
        self.name, self.bias_name, self.fmt = name, bias_name, fmt
        w4 = w if w.dim() == 4 else w[:, :, None, None]
        self.w4, self.shape = w4, tuple(w.shape)
        self.cout, self.cin, self.kh, self.kw = w4.shape
        self.plan = plan if fmt != FMT_F32 else None
        packed = self.plan.add(w4, list(range(self.kh * self.kw)), False) if self.plan is not None else _pack_oihw(w4, fmt)
        self.fwd = ConvW(packed, None if bias is None else bias.contiguous(), self.cin, self.cout, self.kh, self.kw)
        self._dgrad: Dict[Tuple, object] = {}
        if self.plan is not None and need_dx and self.cin % 64 == 0 and self.cout % 64 == 0:
            for py in range(stride):
                for px in range(stride):
                    self.dgrad_tc_weight(stride, pad, py, px)

    def dgrad_simt_weight(self) -> torch.Tensor:
        key = ("simt",)
        if key not in self._dgrad:
            self._dgrad[key] = self.w4.permute(2, 3, 0, 1).reshape(self.kh * self.kw, self.cout, self.cin).contiguous()
        return self._dgrad[key]

    def dgrad_tc_weight(self, stride: int, pad: int, py: int = 0, px: int = 0):
        """Packed weight of the stride-1 convolution over dy that yields the input gradient of parity class
        (py, px) (all pixels when stride == 1).  Returns (ConvW, pad_h, pad_w) or None if the class has no taps."""
        key = ("tc", stride, pad, py, px)
        if key in self._dgrad:
            return self._dgrad[key]

        dys, rs = _dgrad_taps(self.kh, stride, pad, py)
        dxs, ss = _dgrad_taps(self.kw, stride, pad, px)
        if not rs or not ss:
            self._dgrad[key] = None
            return None
        # tap index r' of the sub-kernel reads dy at offset d = r' - pad'  ->  pad' = -d_min; taps must be contiguous in d
        assert dys == list(range(dys[0], dys[0] + len(dys))) and dxs == list(range(dxs[0], dxs[0] + len(dxs)))
        # transposed convolution: O = ci, I = co, taps in increasing-d order
        tap_list = [r * self.kw + s for r in rs for s in ss]
        packed = self.plan.add(self.w4, tap_list, True) if self.plan is not None else _pack_tc(self.w4, self.fmt, tap_list, True)
        cw = ConvW(packed, None, self.cout, self.cin, len(rs), len(ss))
        self._dgrad[key] = (cw, -dys[0], -dxs[0])
        return self._dgrad[key]


class ConvTLayer:
    """nn.ConvTranspose2d(c_in, c_out, kernel 2, stride 2) of the `use_resize_conv=False` decoder (score_unet.py:466-468).
    Its weight [c_in][c_out][2][2] is, read as OIHW, the weight of the stride-2 2x2 convolution C: y-grid -> x-grid whose
    transpose it is: the input gradient is C applied to dy, the weight gradient is C's weight gradient with the roles of
    the tensors swapped."""

    def __init__(self, name: str, w: torch.Tensor, bias: torch.Tensor, fmt: int, bias_name: str):
        self.name, self.bias_name, self.fmt = name, bias_name, fmt
        self.w, self.shape = w.contiguous(), tuple(w.shape)
        self.cin, self.cout = w.shape[0], w.shape[1]
        self.back = ConvW(_pack_oihw(self.w, fmt), None, self.cout, self.cin, 2, 2)          # C: cout channels in, cin out
        self.fwd = pack_transpose(self.w, bias.contiguous(), fmt, lambda a, b: _pack_tc(self.w, fmt, [a * 2 + b], True))


class Tape:
    """Reverse-mode tape over `Act` tensors.  Gradients are keyed by the storage pointer, so views
    (`Act.tokens()`) share their producer's gradient; the tape keeps every activation alive."""

    def __init__(self, fmt: int, device) -> None:
        self.fmt, self.device = fmt, device
        self.steps: List[Callable[[], None]] = []
        self.grads: Dict[int, Act] = {}
        self.keep: List[object] = []

    def record(self, fn: Callable[[], None], *keep) -> None:
        self.steps.append(fn)
        self.keep.extend(keep)

    def pop(self, a: Act) -> Optional[Act]:
        g = self.grads.pop(a.buf.data_ptr(), None)
        if g is not None and (g.n, g.h, g.w, g.c) != (a.n, a.h, a.w, a.c):
            # the gradient was deposited through a view (tokens <-> image): same storage, the consumer's geometry
            assert g.plane == a.plane
            return g.view(a.n, a.h, a.w, a.c)
        return g

    def add(self, a: Act, g: Act) -> None:
        key = a.buf.data_ptr()
        cur = self.grads.get(key)
        if cur is None:
            self.grads[key] = g
        else:
            call("sbgm_add_inplace", cur.ptr, cur.plane, g.ptr, g.plane, self.fmt, cur.plane, _stream())


class TrainKernels:
    """Forward ops that record their backward on a tape."""

    def __init__(self, fmt: int, device, flat_grad: Callable[[str, Tuple[int, ...]], torch.Tensor], params: bool = True) -> None:
        """`flat_grad(name, shape)`: the gradient view of a parameter, reported as produced at once.  `params=False`: only data
        gradients are wanted -- launches whose only product is a parameter gradient are skipped, and `flat_grad` hands out
        scratch for the parameter gradients that kernels produce next to a data gradient."""
        self.fmt, self.device, self.params = fmt, device, params
        self.k = Kernels(fmt, device)
        self.tape: Optional[Tape] = None
        self.param_grad = flat_grad
        self.sync_bn = None          # torch.distributed process group: synchronise BatchNorm statistics over it
        self._scratch: Dict[str, torch.Tensor] = {}

    # -- scratch management --------------------------------------------------------------------
    TICKET_WORDS = 4096        # leading words of a ticketed scratch buffer (kNormTicketWords / kChansumTicketWords)

    def scratch(self, tag: str, floats: int, tickets: bool = False) -> torch.Tensor:
        """`tickets`: the buffer starts with the integer tickets of a last-block reduction (sbgm_norm_backward,
        sbgm_channel_sums): they must be zero before the first use and every launch leaves them zero again."""
        cur = self._scratch.get(tag)
        if cur is None or cur.numel() < floats:
            cur = torch.empty(max(int(floats), 1), dtype=torch.float32, device=self.device)
            if tickets:
                cur[:self.TICKET_WORDS].zero_()
            self._scratch[tag] = cur
        return cur

    def channel_sums(self, dy: Act, dtproj: Optional[torch.Tensor] = None, dbias: Optional[torch.Tensor] = None) -> None:
        """dy summed over the pixels into the rows of `dtproj` (per sample) and / or over the batch too into `dbias`."""
        ws = self.scratch("chansum", _lib.query("sbgm_channel_sums_scratch_floats", dy.n, dy.c), tickets=True)
        call("sbgm_channel_sums", dy.ptr, dy.plane, self.fmt, dy.n, dy.h * dy.w, dy.c, _ptr(dtproj), 0 if dtproj is None else dtproj.stride(0),
             _ptr(dbias), ws.data_ptr(), _stream())

    def wgrad(self, x: Act, dy: Act, dw: torch.Tensor, cin: int, cout: int, kh: int, kw: int, stride: int, pad: int) -> bool:
        """dw [cout][cin][kh][kw] of the convolution x -> dy, on the tensor cores where both channel counts are multiples of 64,
        else on the CUDA cores.  Returns True for the tensor cores."""
        fmt, args = self.fmt, (x.n, x.h, x.w, cin, cout, kh, kw, stride, pad)
        tc = fmt != FMT_F32 and cin % 64 == 0 and cout % 64 == 0
        if tc:
            ws = self.scratch("wgrad", _lib.query("sbgm_conv2d_wgrad_tc_workspace_floats", fmt, *args))
            call("sbgm_conv2d_wgrad_tc", x.ptr, x.plane, dy.ptr, dy.plane, dw.data_ptr(), fmt, *args, ws.data_ptr(), _stream())
        else:
            ws = self.scratch("wgrad", _lib.query("sbgm_conv2d_wgrad_simt_workspace_floats", *args))
            call("sbgm_conv2d_wgrad_simt", x.ptr, x.plane, dy.ptr, dy.plane, dw.data_ptr(), fmt, *args, ws.data_ptr(), _stream())
        return tc

    def grad_like(self, a: Act, zero: bool = False) -> Act:
        g = Act(self.fmt, a.n, a.h, a.w, a.c, self.device)
        if zero:
            g.buf.zero_()
        return g

    # -- convolution ----------------------------------------------------------------------------
    def conv(self, x: Act, layer: ConvLayer, stride: int = 1, pad: int = 0, residual: Optional[Act] = None,
             gn_stats: bool = False, need_dx: bool = True, proj: Optional[torch.Tensor] = None,
             tproj: Optional[torch.Tensor] = None, dtproj: Optional[torch.Tensor] = None, bias_grad: bool = True):
        """`proj`: also emit the nine per-tap partial products of the final 64 -> 1 convolution (returns (y, projected)).
        `tproj` / `dtproj`: per-sample channel offsets added in the epilogue and where their gradient goes.
        `bias_grad=False`: the consumer of y produces this layer's bias gradient as a by-product of its own backward (the
        normalisation behind a decoder convolution, the final 64 -> 1 convolution behind conv_up)."""
        if tproj is not None:
            y, stats = self.k.conv(x, layer.fwd, stride=stride, pad=pad, tproj=tproj), None
        elif proj is not None:
            y, pout = self.k.conv(x, layer.fwd, stride=stride, pad=pad, proj=proj, proj_keep=True)
            stats = None
        else:
            out = self.k.conv(x, layer.fwd, stride=stride, pad=pad, residual=residual, gn_stats=gn_stats)
            y, stats = out if gn_stats else (out, None)
        tape = self.tape

        def backward() -> None:
            dy = tape.pop(y)
            if dy is None:
                return
            self._conv_backward(x, dy, layer, stride, pad, need_dx, bias_grad)
            if residual is not None:
                tape.add(residual, dy)
            if dtproj is not None and self.params:
                self.channel_sums(dy, dtproj=dtproj)

        tape.record(backward, x, y)
        if proj is not None:
            return y, pout
        return (y, stats) if gn_stats else y

    def _conv_backward(self, x: Act, dy: Act, layer: ConvLayer, stride: int, pad: int, need_dx: bool, bias_grad: bool = True) -> None:
        fmt, st = self.fmt, _stream()
        n, h, w = x.n, x.h, x.w
        cin, cout, kh, kw = layer.cin, layer.cout, layer.kh, layer.kw
        if self.params:
            if layer.bias_name is not None and bias_grad:
                self.channel_sums(dy, dbias=self.param_grad(layer.bias_name, (cout,)))
            self.wgrad(x, dy, self.param_grad(layer.name, layer.shape), cin, cout, kh, kw, stride, pad)
        tc = fmt != FMT_F32 and cin % 64 == 0 and cout % 64 == 0          # the data gradient takes the weight gradient's route
        if not need_dx:
            return
        tape = self.tape
        if not tc:
            dx = self.grad_like(x)
            call("sbgm_conv2d_dgrad_simt", dy.ptr, dy.plane, layer.dgrad_simt_weight().data_ptr(), dx.ptr, dx.plane, 0, fmt,
                 n, h, w, cin, cout, kh, kw, stride, pad, st)
            tape.add(x, dx)
            return
        if stride == 1:
            cw, ph, pw = layer.dgrad_tc_weight(1, pad)
            assert ph == pw
            # x already has a gradient from another consumer (the residual branch): it rides in the convolution's epilogue as
            # the residual instead of a separate accumulation pass
            cur = tape.grads.get(x.buf.data_ptr())
            if cur is not None and (cur.n, cur.h, cur.w, cur.c) != (x.n, x.h, x.w, x.c):
                cur = None
            dx = self.k.conv(dy, cw, stride=1, pad=ph, residual=cur)
            assert (dx.h, dx.w) == (h, w)
            if cur is not None:
                tape.grads[x.buf.data_ptr()] = dx
                tape.keep.append(cur)
            else:
                tape.add(x, dx)
            return
        # strided convolution: one stride-1 convolution over dy per input-parity class, scattered into dx
        dx = self.grad_like(x, zero=True)
        for py in range(stride):
            for px in range(stride):
                ent = layer.dgrad_tc_weight(stride, pad, py, px)
                if ent is None:
                    continue
                cw, ph, pw = ent
                ho, wo = (h - py + stride - 1) // stride, (w - px + stride - 1) // stride
                call("sbgm_conv2d_tc_ex", dy.ptr, dy.plane, cw.w.data_ptr(), cw.plane, None, None, 0, 0, None, 0, dx.ptr, dx.plane, fmt,
                     dy.n, dy.h, dy.w, cout, cin, cw.kh, cw.kw, 1, ph, pw, ho, wo, h, w, stride, py, px, ACT_NONE, None, 0, st)
        tape.add(x, dx)

    # -- normalisation ------------------------------------------------------------------------------
    def _norm(self, x: Act, stats: torch.Tensor, mode: int, groups: int, gamma, beta, gamma_name, beta_name, add: Optional[Act],
              tproj: Optional[torch.Tensor], dtproj: Optional[torch.Tensor], tproj_pre: int, act: int,
              prev_bias: Optional[str] = None) -> Act:
        fmt = self.fmt
        y = x.like()
        hw = x.h * x.w
        call("sbgm_norm_apply", x.ptr, x.plane, stats.data_ptr(), mode, groups, _ptr(gamma), _ptr(beta),
             None if add is None else add.ptr, 0 if add is None else add.plane, _ptr(tproj),
             tproj.stride(0) if tproj is not None else 0, tproj_pre, act, y.ptr, y.plane, fmt, x.n, hw, x.c, _stream())
        tape = self.tape

        def backward() -> None:
            dy = tape.pop(y)
            if dy is None:
                return
            dx = self.grad_like(x)
            dadd = self.grad_like(x) if add is not None else None
            dg = self.param_grad(gamma_name, (x.c,)) if gamma_name else None
            db = self.param_grad(beta_name, (x.c,)) if beta_name else None
            dprev = self.param_grad(prev_bias, (x.c,)) if prev_bias else None      # bias gradient of the convolution that made x
            ws = self.scratch("norm_bwd", _lib.query("sbgm_norm_backward_scratch_floats", x.n, x.c), tickets=True)

            def run(stage: int, sums_all: Optional[torch.Tensor], n_all: int) -> None:
                call("sbgm_norm_backward", dy.ptr, dy.plane, x.ptr, x.plane, stats.data_ptr(), mode, groups, _ptr(gamma), _ptr(beta),
                     None if add is None else add.ptr, 0 if add is None else add.plane, _ptr(tproj),
                     tproj.stride(0) if tproj is not None else 0, tproj_pre, act, dx.ptr, dx.plane,
                     None if dadd is None else dadd.ptr, 0 if dadd is None else dadd.plane, _ptr(dg), _ptr(db), _ptr(dprev),
                     _ptr(dtproj), dtproj.stride(0) if dtproj is not None else 0, fmt, x.n, hw, x.c, ws.data_ptr(), stage,
                     _ptr(sums_all), n_all, _stream())

            if mode == 0 and self.sync_bn is not None:
                # synchronised BatchNorm: the projection terms need the sums over the WHOLE batch
                import torch.distributed as dist
                run(1, None, 0)
                off = _lib.query("sbgm_norm_backward_sums_offset", x.n, x.c)
                local = ws[off:off + _lib.query("sbgm_norm_backward_sums_floats", x.n, x.c)]
                world = dist.get_world_size(self.sync_bn)
                sums_all = torch.empty(world * local.numel(), dtype=torch.float32, device=self.device)
                dist.all_gather_into_tensor(sums_all, local, group=self.sync_bn)
                run(2, sums_all, world * x.n)
            else:
                run(0, None, 0)
            tape.add(x, dx)
            if add is not None:
                tape.add(add, dadd)

        tape.record(backward, x, y, stats)
        return y

    def batchnorm(self, x: Act, bn: dict, train: bool, act: int = ACT_NONE, residual: Optional[Act] = None,
                  tproj: Optional[torch.Tensor] = None, dtproj: Optional[torch.Tensor] = None) -> Act:
        """nn.BatchNorm2d (+residual, ReLU, then the time projection).  train=True: batch statistics and
        running-stat update (torchvision resnet.py:89-103 in .train()); else the running statistics as constants."""
        c, hw = x.c, x.h * x.w
        stats = torch.empty((c, 2), dtype=torch.float32, device=self.device)
        if train:
            chunks = _lib.query("sbgm_norm_partials_chunks", hw, c)
            part = torch.empty((x.n, chunks, c, 2), dtype=torch.float32, device=self.device)
            call("sbgm_norm_partials", x.ptr, x.plane, self.fmt, x.n, hw, c, c, part.data_ptr(), _stream())
            n_all = x.n
            if self.sync_bn is not None:
                # whole-batch statistics: gather every rank's partial sums (rank-major = the unsharded sample order, so the
                # finalised statistics are bit-identical to a single-GPU run of the full batch)
                import torch.distributed as dist
                world = dist.get_world_size(self.sync_bn)
                gathered = torch.empty((world * x.n, chunks, c, 2), dtype=torch.float32, device=self.device)
                dist.all_gather_into_tensor(gathered, part, group=self.sync_bn)
                part, n_all = gathered, world * x.n
            call("sbgm_bn_stats_finalize", part.data_ptr(), chunks, n_all, hw, c, BN_EPS, BN_MOMENTUM, stats.data_ptr(),
                 bn["running_mean"].data_ptr(), bn["running_var"].data_ptr(), _stream())
            mode = 0
        else:
            stats[:, 0] = bn["running_mean"]
            stats[:, 1] = torch.rsqrt(bn["running_var"] + BN_EPS)
            mode = 2
        return self._norm(x, stats, mode, c, bn["weight"], bn["bias"], bn["weight_name"], bn["bias_name"], residual, tproj, dtproj, 0, act)

    def groupnorm(self, x: Act, gamma, beta, gamma_name, beta_name, groups: int, act: int = ACT_NONE, skip: Optional[Act] = None,
                  tproj: Optional[torch.Tensor] = None, dtproj: Optional[torch.Tensor] = None, fused=None,
                  prev_bias: Optional[str] = None) -> Act:
        hw = x.h * x.w
        stats = torch.empty((x.n, groups, 2), dtype=torch.float32, device=self.device)
        if fused is not None and (x.c // 8) % groups == 0:
            part, chunks = fused
            pgroups = x.c // 8
        else:
            chunks, pgroups = _lib.query("sbgm_norm_partials_chunks", hw, x.c), groups
            part = torch.empty((x.n, chunks, groups, 2), dtype=torch.float32, device=self.device)
            call("sbgm_norm_partials", x.ptr, x.plane, self.fmt, x.n, hw, x.c, groups, part.data_ptr(), _stream())
        call("sbgm_gn_stats_finalize", part.data_ptr(), chunks, pgroups, groups, x.n, hw, x.c, GN_EPS, stats.data_ptr(), _stream())
        return self._norm(x, stats, 1, groups, gamma, beta, gamma_name, beta_name, skip, tproj, dtproj, 1, act, prev_bias)

    def layernorm(self, x: Act, gamma, beta, gamma_name, beta_name) -> Act:
        y = self.k.layernorm(x, gamma, beta)
        tape = self.tape

        def backward() -> None:
            dy = tape.pop(y)
            if dy is None:
                return
            dx = self.grad_like(x)
            rows = x.n * x.h * x.w
            ws = self.scratch("ln_bwd", _lib.query("sbgm_layernorm_backward_scratch_floats", x.c))
            call("sbgm_layernorm_backward", dy.ptr, dy.plane, x.ptr, x.plane, gamma.data_ptr(), LN_EPS, dx.ptr, dx.plane,
                 self.param_grad(gamma_name, (x.c,)).data_ptr(), self.param_grad(beta_name, (x.c,)).data_ptr(), self.fmt, rows, x.c,
                 ws.data_ptr(), _stream())
            tape.add(x, dx)

        tape.record(backward, x, y)
        return y

    def activation(self, x: Act, act: int) -> Act:
        y = x.like()
        call("sbgm_act_forward", x.ptr, x.plane, y.ptr, y.plane, self.fmt, x.plane, act, _stream())
        tape = self.tape

        def backward() -> None:
            dy = tape.pop(y)
            if dy is None:
                return
            dx = self.grad_like(x)
            call("sbgm_act_backward", dy.ptr, dy.plane, x.ptr, x.plane, dx.ptr, dx.plane, self.fmt, x.plane, act, _stream())
            tape.add(x, dx)

        tape.record(backward, x, y)
        return y

    def conv_transpose2x(self, x: Act, layer: ConvTLayer) -> Act:
        y = self.k.conv_transpose2x(x, layer.fwd)
        tape = self.tape

        def backward() -> None:
            dy = tape.pop(y)
            if dy is None:
                return
            if self.params:
                self.channel_sums(dy, dbias=self.param_grad(layer.bias_name, (layer.cout,)))
                # C: input dy-grid (cout channels), output x-grid
                self.wgrad(dy, x, self.param_grad(layer.name, layer.shape), layer.cout, layer.cin, 2, 2, 2, 0)
            tape.add(x, self.k.conv(dy, layer.back, stride=2, pad=0))

        tape.record(backward, x, y)
        return y

    def upsample2x(self, x: Act) -> Act:
        y = self.k.upsample2x(x)
        tape = self.tape

        def backward() -> None:
            dy = tape.pop(y)
            if dy is None:
                return
            dx = self.grad_like(x)
            call("sbgm_upsample2x_backward", dy.ptr, dy.plane, dx.ptr, dx.plane, self.fmt, x.n, x.h, x.w, x.c, _stream())
            tape.add(x, dx)

        tape.record(backward, x, y)
        return y

    def attention_core(self, qkv: Act, b: int, s: int, c: int, heads: int) -> Act:
        y = self.k.attention_core(qkv, b, s, c, heads)
        tape = self.tape

        def backward() -> None:
            dy = tape.pop(y)
            if dy is None:
                return
            dqkv = self.grad_like(qkv)
            ws = self.scratch("attn_bwd", _lib.query("sbgm_attention_backward_scratch_floats", b, s, c, heads))
            call("sbgm_attention_backward", qkv.ptr, qkv.plane, y.ptr, y.plane, dy.ptr, dy.plane, dqkv.ptr, dqkv.plane, self.fmt, b, s, c,
                 heads, ws.data_ptr(), _stream())
            tape.add(qkv, dqkv)

        tape.record(backward, qkv, y)
        return y


def _attn_layers(sd, keys: AttnKeys, fmt: int, plan: PackPlan) -> AttnKeys:
    """An attention block under its layout's field names: ConvLayers, and (gamma, beta, gamma name, beta name) per LayerNorm."""
    lin = lambda a: ConvLayer(a.weight, sd[a.weight], sd[a.bias], fmt, a.bias, plan=plan)
    ln = lambda a: (sd[a.weight], sd[a.bias], *a)
    return AttnKeys(ln(keys.ln1), lin(keys.in_proj), lin(keys.out_proj), ln(keys.ln2), lin(keys.ff0), lin(keys.ff2))


def _attention_block(tk: TrainKernels, aw: AttnKeys, heads: int, x: Act) -> Act:
    """ImageSelfAttention.forward (score_unet.py:136-148) with its backward recorded."""
    tok = x.tokens()
    b, s, c = x.n, x.h * x.w, x.c
    h1 = tk.layernorm(tok, *aw.ln1)
    qkv = tk.conv(h1, aw.in_proj)
    att = tk.attention_core(qkv, b, s, c, heads)
    h = tk.conv(att, aw.out_proj, residual=tok)
    g = tk.layernorm(h, *aw.ln2)
    g1 = tk.conv(g, aw.ff0)
    g2 = tk.activation(g1, ACT_GELU)
    return tk.conv(g2, aw.ff2, residual=h).view(x.n, x.h, x.w, x.c)


class TrainEngine:
    """One forward + backward of the score-UNet for the DSM training step.

    `params` maps state-dict names to the live parameter / buffer tensors (fp32, CUDA).  BatchNorm running
    statistics are updated in place when `bn_train` is set."""

    def __init__(self, params: Dict[str, torch.Tensor], spec: UNetSpec, precision: str, device, bn_train: bool,
                 encoder_only: bool = False, input_grads: Tuple[bool, bool] = (False, False), param_grads: bool = True) -> None:
        """`encoder_only`: `params` is the standalone Encoder's own state dict and `forward` returns its five feature maps
        (`Encoder.forward` in .train(): batch statistics, running statistics updated; nothing is differentiated).
        `input_grads` = (x, planes): backward also returns the gradient of x / of the conditioning planes (keys DX, DPLANES).
        `param_grads=False`: backward computes data gradients only -- no flat gradient buffer, no weight-gradient launches, no
        gradient exchange."""
        device = engine_device(precision, device)
        self.spec, self.device, self.fmt, self.bn_train = spec, device, TRAIN_PRECISIONS[precision], bn_train
        self.input_grads, self.param_grads = tuple(bool(v) for v in input_grads), param_grads
        self.encoder_only = encoder_only
        self.enc_layout = encoder_layout(spec, "") if encoder_only else encoder_layout(spec)
        self.dec_layout = None if encoder_only else decoder_layout(spec)
        self.sd = {k: v.detach() for k, v in params.items()}
        for k, v in self.sd.items():
            if v.is_floating_point() and (v.dtype != torch.float32 or not v.is_cuda):
                raise RuntimeError(f"parameter {k} must be fp32 on CUDA for the training path, got {v.dtype} on {v.device}")
        # flat gradient buffer: parameters in state-dict order, each gradient a view (parallel.py all-reduces it in place)
        names = [k for k, v in params.items() if isinstance(v, torch.nn.Parameter) or v.requires_grad]
        self.grad_names = flat_order(names)
        self.offsets: Dict[str, Tuple[int, int]] = {}
        off = 0
        for k in self.grad_names:
            self.offsets[k] = (off, self.sd[k].numel())
            off += (self.sd[k].numel() + 63) // 64 * 64
        self.flat_numel = off
        self.flat: Optional[torch.Tensor] = None
        self.touched: Dict[str, torch.Tensor] = {}
        self._sink: Dict[str, torch.Tensor] = {}     # parameter-gradient by-products when param_grads is off
        self.tk = TrainKernels(self.fmt, device, self._param_grad, params=param_grads)
        self.grad_sync = None      # parallel.GradSync or None
        with torch.cuda.device(device), torch.no_grad():
            self._pack()

    # -- parameters -------------------------------------------------------------------------------
    def _param_grad(self, name: str, shape: Tuple[int, ...]) -> torch.Tensor:
        if not self.param_grads:
            g = self._sink.get(name)
            if g is None:
                g = self._sink[name] = torch.empty(shape, dtype=torch.float32, device=self.device)
            return g
        off, numel = self.offsets[name]
        g = self.flat[off:off + numel].view(shape)
        self.touched[name] = g
        return g

    def _conv(self, wname: str, bname: Optional[str] = None, stride: int = 1, pad: int = 0) -> ConvLayer:
        return ConvLayer(wname, self.sd[wname], None if bname is None else self.sd[bname], self.fmt, bname, plan=self.plan,
                         stride=stride, pad=pad)

    def _conv_bn(self, s: ConvBN, stride: int, pad: int) -> ConvBN:
        bn = {field: self.sd[key] for field, key in s.bn._asdict().items()}          # weight, bias, running_mean, running_var
        return ConvBN(self._conv(s.conv, stride=stride, pad=pad), dict(bn, weight_name=s.bn.weight, bias_name=s.bn.bias))

    def _up(self, s: Affine):
        return (self._conv(*s, 1, 1) if self.spec.use_resize_conv else
                ConvTLayer(s.weight, self.sd[s.weight], self.sd[s.bias], self.fmt, s.bias))

    def _dec_block(self, s: DecBlock) -> DecBlock:
        norm = lambda a: (None,) * 4 if a is None else (self.sd[a.weight], self.sd[a.bias], *a)      # gamma, beta and their names
        return s._replace(conv_up=self._up(s.conv_up), conv=self._conv(*s.conv, 1, 1), n1=norm(s.n1), n2=norm(s.n2),
                          attn=None if s.attn is None else _attn_layers(self.sd, s.attn, self.fmt, self.plan))

    def _pack(self) -> None:
        sd, spec, fmt, enc = self.sd, self.spec, self.fmt, self.enc_layout
        self.plan = PackPlan(fmt)
        w1 = sd[enc.stem]
        self.cin = w1.shape[1]
        self.stem_w = stem_matrix(w1)
        if fmt != FMT_F32:   # tensor-core stem: 1x1 convolution over the im2col tensor; [co][ci*64 + tap] IS conv1.weight's OIHW order
            self.stem_layer = ConvLayer(enc.stem, w1.reshape(64, self.cin * 64, 1, 1), None, fmt, plan=self.plan, need_dx=False)
            self.stem_layer.shape = tuple(w1.shape)
        if any(self.input_grads) and fmt != FMT_F32:
            self.stem_dgrad_w = stem_dgrad_weight(self.plan, w1)
        self.conv2, self.bn1 = self._conv_bn(enc.conv2, 2, 3)
        self.layers = [[s._replace(down=None if s.down is None else self._conv_bn(s.down, s.stride, 0), c1=self._conv_bn(s.c1, s.stride, 1),
                                   c2=self._conv_bn(s.c2, 1, 1)) for s in stage] for stage in enc.stages]
        self.enc_attn = {i: _attn_layers(sd, keys, fmt, self.plan) for i, keys in enc.attn.items()}
        # time projector: same packing as inference (engine.TimeProjector) plus the names for the gradients
        self.tp_heads = enc.heads + (() if self.encoder_only else tuple(s.head for s in self.dec_layout.blocks))
        self.tp = TimeProjector(self.device, spec.time_embedding)
        self.tp.add_heads(self.tp_heads, sd.__getitem__)
        if enc.label_emb is not None:
            self.tp.label_emb = sd[enc.label_emb].contiguous()
        self.tp.finalize()
        self.act = ACTS[spec.activation]
        if (dec := self.dec_layout) is not None:
            self.dec_blocks = [self._dec_block(s) for s in dec.blocks]
            self.final_up = self._up(dec.final_up)
            wf = sd[dec.final_conv.weight]
            if wf.shape[0] != 1:
                raise NotImplementedError("the training path supports output_channels == 1 (the reference's only configuration)")
            self.final_w = final_matrix(wf)
            self.final_b = sd[dec.final_conv.bias].contiguous()
        self.plan.run()            # every forward / data-gradient pack of the step: one batched launch

    # -- forward ----------------------------------------------------------------------------------------
    def forward(self, x: torch.Tensor, t: Optional[torch.Tensor], y: Optional[torch.Tensor], planes: Optional[torch.Tensor],
                inv_std: Optional[torch.Tensor], *, sampler: Optional[dict] = None) -> torch.Tensor:
        """`sampler` (score_sampling._TrainModeStep: a sampler step with batch-statistics BatchNorm, captured in a CUDA graph):
        dict(tproj=[n, c_total] time projections already computed for the step, inv_std=engine.InvStd of the step table's 1/std
        column, dst=output tensor); no gradient buffer is set up and the recorded tape is dropped."""
        tk, fmt, dev = self.tk, self.fmt, self.device
        tape = Tape(fmt, dev)
        tk.tape = tape
        self.tape = tape
        self._sampler = sampler
        self.touched = {}
        n, _, h, w = x.shape
        cc = self.cin - 1
        if cc > 0 and (planes is None or planes.shape[1] != cc):
            raise AssertionError(f"encoder expects {cc} conditioning channels")
        yy = None if y is None else y.reshape(-1).to(device=dev, dtype=torch.int64).contiguous()
        if sampler is not None:
            self.flat = None
            tproj = sampler["tproj"]
            dtproj = tproj                     # never written: no backward runs on a sampler step
        else:
            self.flat = torch.zeros(self.flat_numel, dtype=torch.float32, device=dev) if self.param_grads else None
            t = t.reshape(-1).to(device=dev, dtype=torch.float32).contiguous()
            tproj = self.tp(t, yy)
            dtproj = torch.zeros_like(tproj)
        tape.keep += [tproj, t, yy, x, planes]
        col = lambda table, name: self.tp.cols(table, name)

        self._time = (t, yy, dtproj)
        # Encoder.conv1 + time projection 0 (score_unet.py:310-314)
        t0 = col(tproj, "enc0")
        self._input_grads = {}
        if fmt != FMT_F32:
            xcol = tk.k.stem_im2col(x, planes, 0, self.cin, cc)
            f1 = tk.conv(xcol, self.stem_layer, need_dx=False, tproj=t0, dtproj=col(dtproj, "enc0"))
            if any(self.input_grads):
                # recorded after the stem's own step, so it runs first in backward and reads df before that step consumes it
                tape.record(lambda: self._stem_dgrad(tape.grads.get(f1.buf.data_ptr()), x, planes))
            return self._forward_rest(f1, tproj, dtproj, inv_std, n)
        f1 = Act(fmt, n, h // 2, w // 2, 64, dev)
        call("sbgm_stem_conv", x.data_ptr(), _ptr(planes), 1 if planes is None else planes.shape[0], cc, 0, self.cin,
             self.stem_w.data_ptr(), None, 0, t0.data_ptr(), t0.stride(0), f1.ptr, f1.plane, fmt, n, h, w, _stream())

        def stem_backward() -> None:
            df = tape.pop(f1)
            if df is None:
                return
            self._stem_dgrad(df, x, planes)
            if not self.param_grads:
                return
            tk.channel_sums(df, dtproj=col(dtproj, "enc0"))
            dw = self._param_grad(self.enc_layout.stem, (64, self.cin, 8, 8))
            ws2 = tk.scratch("stem", _lib.query("sbgm_stem_wgrad_workspace_floats", self.cin))
            call("sbgm_stem_wgrad", x.data_ptr(), _ptr(planes), 1 if planes is None else planes.shape[0], cc, df.ptr, df.plane, fmt,
                 dw.data_ptr(), n, h, w, ws2.data_ptr(), _stream())

        tape.record(stem_backward, f1)
        return self._forward_rest(f1, tproj, dtproj, inv_std, n)

    def _stem_dgrad(self, df: Optional[Act], x: torch.Tensor, planes: Optional[torch.Tensor]) -> None:
        """Encoder.conv1's data gradient: the requested ones of dx [n, 1, h, w] and dplanes [np, cc, h, w] (fp32) into
        self._input_grads (zeros when nothing reached the stem)."""
        want_x, want_planes = self.input_grads
        want_planes = want_planes and planes is not None
        if not (want_x or want_planes):
            return
        dx = torch.empty_like(x) if want_x else None
        dpl = torch.empty_like(planes) if want_planes else None
        if df is None:
            for g in (dx, dpl):
                if g is not None:
                    g.zero_()
        else:
            n, _, h, w = x.shape
            np_, cc = (1, 0) if planes is None else (planes.shape[0], planes.shape[1])
            ws = self.tk.scratch("stem_dgrad", _lib.query("sbgm_stem_dgrad_workspace_floats", np_, cc, n, h, w))
            if self.fmt == FMT_F32:
                call("sbgm_stem_dgrad_simt", df.ptr, df.plane, self.fmt, self.sd[self.enc_layout.stem].data_ptr(), _ptr(dx), _ptr(dpl),
                     np_, cc, n, h, w, ws.data_ptr(), _stream())
            else:
                wt = self.stem_dgrad_w
                call("sbgm_stem_dgrad_tc", df.ptr, df.plane, self.fmt, wt.data_ptr(), wt.stride(1), _ptr(dx), _ptr(dpl), np_, cc, n, h, w,
                     ws.data_ptr(), _stream())
        if dx is not None:
            self._input_grads[DX] = dx
        if dpl is not None:
            self._input_grads[DPLANES] = dpl

    def _forward_rest(self, f1: Act, tproj: torch.Tensor, dtproj: torch.Tensor, inv_std: Optional[torch.Tensor], n: int) -> torch.Tensor:
        tk, fmt, dev, tape = self.tk, self.fmt, self.device, self.tape
        col = lambda table, name: self.tp.cols(table, name)
        fmaps = [f1]
        hcur = tk.batchnorm(tk.conv(f1, self.conv2, stride=2, pad=3), self.bn1, self.bn_train, act=ACT_RELU)
        for li, blocks in enumerate(self.layers, start=1):
            for bi, blk in enumerate(blocks):
                last = bi == len(blocks) - 1
                if blk.down is not None:
                    idn = tk.batchnorm(tk.conv(hcur, blk.down.conv, stride=blk.stride, pad=0), blk.down.bn, self.bn_train)
                else:
                    idn = hcur
                mid = tk.batchnorm(tk.conv(hcur, blk.c1.conv, stride=blk.stride, pad=1), blk.c1.bn, self.bn_train, act=ACT_RELU)
                hcur = tk.batchnorm(tk.conv(mid, blk.c2.conv, stride=1, pad=1), blk.c2.bn, self.bn_train, act=ACT_RELU, residual=idn,
                                    tproj=col(tproj, f"enc{li}") if last else None, dtproj=col(dtproj, f"enc{li}") if last else None)
            if li in self.enc_attn:
                hcur = _attention_block(tk, self.enc_attn[li], self.spec.n_heads, hcur)
            fmaps.append(hcur)
        if self.encoder_only:                  # standalone Encoder.forward: the feature maps are the result, no backward follows
            self.tape = tk.tape = None
            self._final = self._time = self._sampler = None
            return fmaps

        # Decoder (score_unet.py:733-758)
        rev = list(reversed(fmaps))
        out = rev[0]
        for i, blk in enumerate(self.dec_blocks):
            # the two convolutions' bias gradients come out of the normalisation backward behind them (closed form)
            if self.spec.use_resize_conv:
                a, st1 = tk.conv(tk.upsample2x(out), blk.conv_up, pad=1, gn_stats=True, bias_grad=False)
                a = tk.groupnorm(a, *blk.n1, groups=blk.g1, fused=st1, prev_bias=blk.conv_up.bias_name)
            else:
                a = tk.groupnorm(tk.conv_transpose2x(out, blk.conv_up), *blk.n1, groups=blk.g1)
            b, st2 = tk.conv(a, blk.conv, pad=1, gn_stats=True, bias_grad=False)
            skip = rev[i + 1]
            if (skip.n, skip.h, skip.w, skip.c) != (b.n, b.h, b.w, b.c):
                raise AssertionError(f"prev_fmap shape {(skip.n, skip.c, skip.h, skip.w)} must match output shape {(b.n, b.c, b.h, b.w)}")
            out = tk.groupnorm(b, *blk.n2, groups=blk.g2, act=self.act, skip=skip, tproj=col(tproj, blk.head.name),
                               dtproj=col(dtproj, blk.head.name), fused=st2, prev_bias=blk.conv.bias_name)
            if blk.attn is not None:
                out = _attention_block(tk, blk.attn, self.spec.n_heads, out)
        smp = getattr(self, "_sampler", None)
        res = smp["dst"] if smp is not None else torch.empty((n, 1, 2 * out.h, 2 * out.w), dtype=torch.float32, device=dev)
        # 1 / std per member (training) or per sampler step (row of the step table selected by the device step counter)
        iv = InvStd(inv_std) if smp is None else smp["inv_std"]
        pr = None
        if not self.spec.use_resize_conv:
            a = tk.conv_transpose2x(out, self.final_up)
        else:
            up = tk.upsample2x(out)
            if fmt != FMT_F32 and tk.k._c64_ok(up, self.final_up.fwd, 1, 1):
                # the 64 -> 1 convolution rides in conv_up's epilogue (projection); conv_up's output is kept for the backward
                a, pr = tk.conv(up, self.final_up, pad=1, proj=self.final_w[0], bias_grad=not self._final_bias_fused())
            else:
                a = tk.conv(up, self.final_up, pad=1, bias_grad=not self._final_bias_fused())
        if pr is None:
            tk.k.final_conv(a, self.final_w, self.final_b, iv, res)
        else:
            tk.k.final_gather(pr, self.final_b, iv, res)
        if smp is not None:                    # a sampler step: nothing will run backward -- drop the tape and its activations
            self.tape = tk.tape = None
            self._final = self._time = self._sampler = None
            return res
        self._final = (a, inv_std)
        return res

    def _final_bias_fused(self) -> bool:
        """final_layer.conv_up's bias gradient is a by-product of the final convolution's backward (sbgm_final_conv_backward's
        dbias_up) when conv_up is the resize-convolution and its channel-vector count is a power of two."""
        vecs = self.final_w.shape[2] // 8
        return self.spec.use_resize_conv and self.final_w.shape[2] % 8 == 0 and 8 <= vecs <= 32 and vecs & (vecs - 1) == 0

    # -- backward ----------------------------------------------------------------------------------------
    def backward(self, dscore: torch.Tensor) -> Dict[str, torch.Tensor]:
        """dscore: gradient of the loss w.r.t. the network output [n, 1, h, w] (fp32).  Returns {name: grad}."""
        tk, tape, fmt = self.tk, self.tape, self.fmt
        a, inv_std = self._final
        t, yy, dtproj = self._time
        params = self.param_grads
        dscore = dscore.to(device=self.device, dtype=torch.float32).contiguous()
        da = tk.grad_like(a)
        dwf = self._param_grad(self.dec_layout.final_conv.weight, (1, a.c, 3, 3))
        dbf = self._param_grad(self.dec_layout.final_conv.bias, (1,))
        dbu = self._param_grad(self.final_up.bias_name, (a.c,)) if self._final_bias_fused() else None
        ws = tk.scratch("final", _lib.query("sbgm_final_conv_backward_scratch_floats", a.c))
        call("sbgm_final_conv_backward", dscore.data_ptr(), _ptr(inv_std), a.ptr, a.plane, fmt, self.final_w.data_ptr(), da.ptr, da.plane,
             dwf.data_ptr(), dbf.data_ptr(), _ptr(dbu), a.n, a.h, a.w, a.c, ws.data_ptr(), _stream())
        tape.add(a, da)
        sync = self.grad_sync if params else None
        if sync is not None:
            sync.begin(self.flat, [(k, *self.offsets[k]) for k in self.grad_names])
        reported = 0
        for fn in reversed(tape.steps):
            fn()
            if sync is not None and len(self.touched) > reported:
                new = list(self.touched)[reported:]
                reported = len(self.touched)
                sync.progress(new)
        if not params:
            grads = dict(self._input_grads)
            self.tape = tk.tape = None
            self._final = self._time = None
            return grads
        # time embedding: one launch set for all nine projections (+ label embedding)
        fw, pw, pb, ps = self.tp._packed
        rows = t.numel()
        # flat_order lays the nine projection weights, then the nine biases, out in head order: when they are contiguous (every
        # size is a multiple of the 64-element padding) the kernel writes the flat buffer directly, no per-head copies
        wviews = [self._param_grad(h.weight, tuple(self.sd[h.weight].shape)) for h in self.tp_heads]
        bviews = [self._param_grad(h.bias, tuple(self.sd[h.bias].shape)) for h in self.tp_heads]
        in_place = all(b.data_ptr() == a.data_ptr() + a.nbytes for views in (wviews, bviews) for a, b in zip(views, views[1:]))
        dpw = wviews[0] if in_place else torch.empty_like(pw)
        dpb = bviews[0] if in_place else torch.empty_like(pb)
        lab = self.enc_layout.label_emb
        dlab = self._param_grad(lab, tuple(self.sd[lab].shape)) if (lab and yy is not None) else None
        ws = tk.scratch("time", _lib.query("sbgm_time_embed_backward_scratch_floats", fw.shape[0], self.tp.te, rows))
        call("sbgm_time_embed_backward", dtproj.data_ptr(), t.data_ptr(), _ptr(yy), fw.data_ptr(), fw.shape[0], self.tp.te,
             _ptr(self.tp.label_emb) if yy is not None else None, 0 if dlab is None else dlab.shape[0], pw.data_ptr(), ps.data_ptr(),
             self.tp.c_total, rows, dpw.data_ptr(), dpb.data_ptr(), _ptr(dlab), ws.data_ptr(), _stream())
        if not in_place:
            sizes = [len(bv) for bv in bviews]
            for wv, bv, dw, db in zip(wviews, bviews, dpw.split(sizes), dpb.split(sizes)):
                wv.copy_(dw)
                bv.copy_(db)
        if sync is not None:
            sync.progress(list(self.touched)[reported:])
            sync.finish()
        grads = dict(self.touched, **self._input_grads)
        self.tape = None
        tk.tape = None
        self._final = self._time = None
        return grads


def flat_order(names: Sequence[str]) -> List[str]:
    """Order of the parameters in the flat gradient buffer: the order in which the FORWARD pass uses them, so that backward
    produces gradients from the END of the buffer down and the bucketed all-reduce (parallel.GradBucketer walks buckets from
    the end) can start while backward is still running.  The time projections and the label embedding come first: their
    gradients are the last thing backward produces (one launch for all nine heads, TrainEngine.backward).  Within a stage the
    state-dict order is kept (stable sort)."""
    def stage(k: str):
        if k.endswith("label_emb.weight"):
            return -3
        if "time_projection_layer" in k:      # weights first, then biases, each in head order (encoder 0..4, decoder blocks):
            return -2 if k.endswith(".weight") else -1     # one contiguous range each (TrainEngine.backward writes them in place)
        if k.startswith("encoder."):
            rest = k[len("encoder."):]
            if rest.startswith("conv1."):
                return 1
            if rest.startswith(("conv2.", "bn1.")):
                return 2
            for li in range(1, 5):
                if rest.startswith(f"layer{li}."):
                    return 1 + 2 * li              # 3, 5, 7, 9
            for li in range(5):
                if rest.startswith(f"attention_layers.{li}."):
                    return 2 + 2 * li              # after its stage: 8 (index 3), 10 (index 4)
            return 2
        if k.startswith("decoder.residual_layers."):
            return 20 + int(k.split(".")[2])
        if k.startswith("decoder.final_layer."):
            return 40
        return 50
    return sorted(names, key=stage)


class _InFlight:
    """Clears the runner's busy flag when the autograd node that owns it is dropped without a backward."""

    def __init__(self, runner: "TrainRunner") -> None:
        self.runner = runner

    def release(self) -> None:
        if self.runner is not None:
            self.runner.busy = False
            self.runner = None

    def __del__(self) -> None:
        self.release()


class TrainRunner:
    """Runs `TrainEngine` eagerly for the first steps, then as two captured CUDA graphs (forward, backward).

    A training step is ~1 500 kernel launches sequenced from Python; replaying it from a graph removes the host
    from the step (the reference's torch-eager loop is launch-bound in the same way).  Everything a step reads that
    changes between steps lives in static device buffers: the inputs are copied in, parameters are updated in place
    by the optimizer (the graph re-packs them), BatchNorm running statistics are updated in place by the graph.
    The runner is keyed (by the caller) on shapes, precision, mode and parameter storage; a second forward while a
    step is in flight, or graphs disabled (SBGM_B200_TRAIN_GRAPHS=0), falls back to the eager engine."""

    WARMUP = 2

    def __init__(self, make_engine: Callable[[], "TrainEngine"], use_graphs: bool = True) -> None:
        self.make_engine, self.use_graphs = make_engine, use_graphs
        self.calls = 0
        self.busy = False
        self.eng: Optional[TrainEngine] = None
        self.g_fwd = self.g_bwd = None
        self.static: Dict[str, Optional[torch.Tensor]] = {}
        self.out: Optional[torch.Tensor] = None
        self.grads: Optional[Dict[str, torch.Tensor]] = None
        self.keep: list = []

    def _capture_failed(self, exc: Exception) -> None:
        import warnings
        self.capture_failures = getattr(self, "capture_failures", 0) + 1
        self.eng = self.g_fwd = self.g_bwd = self.out = self.grads = None
        self.static, self.keep = {}, []
        try:
            torch.cuda.synchronize()
        except Exception:
            pass
        if self.capture_failures >= 3:
            self.use_graphs = False
        warnings.warn(f"sbgm_danra_b200: CUDA-graph capture of the training step failed ({type(exc).__name__}: {str(exc)[:200]}); "
                      + ("staying on the eager launch sequence" if not self.use_graphs else "this step runs eagerly, capture will be retried"))

    def _backward_capture_failed(self, exc: Exception, inflight: "_InFlight", dout: torch.Tensor) -> Dict[str, torch.Tensor]:
        """This step's forward graph has run, its backward could not be captured (and a half-walked tape cannot be resumed):
        drop both graphs and redo the step on the eager launch sequence from the static inputs -- same gradients; with
        train-mode BatchNorm the running statistics see this batch twice.  With a gradient exchange attached the ranks would
        no longer issue the same collectives, so there the failure is raised."""
        static, sync = self.static, (None if self.eng is None else self.eng.grad_sync)
        self._capture_failed(exc)
        inflight.release()
        if sync is not None and sync.world > 1:
            raise RuntimeError("sbgm_danra_b200: capturing the backward graph of a data-parallel training step failed; "
                               "set SBGM_B200_TRAIN_GRAPHS=0 to train on the eager launch sequence") from exc
        eng = self._engine(sync)
        eng.forward(*(static[k] for k in ("x", "t", "y", "planes", "inv_std")))
        return eng.backward(dout)

    @staticmethod
    def _copy_in(dst: Optional[torch.Tensor], src: Optional[torch.Tensor]) -> None:
        if dst is not None:
            dst.copy_(src)

    def _engine(self, grad_sync) -> "TrainEngine":
        eng = self.make_engine()
        eng.grad_sync = grad_sync
        if grad_sync is not None and getattr(grad_sync, "sync_bn", False) and grad_sync.world > 1:
            import torch.distributed as dist
            eng.tk.sync_bn = grad_sync.group if grad_sync.group is not None else dist.group.WORLD
        return eng

    def forward(self, x, t, y, planes, inv_std, grad_sync):
        self.calls += 1
        graph_ok = self.use_graphs and self.calls > self.WARMUP and not self.busy
        if not graph_ok:
            eng = self._engine(grad_sync)
            return eng.forward(x, t, y, planes, inv_std), ("eager", eng)
        ins = dict(x=x, t=t, y=y, planes=planes, inv_std=inv_std)
        if self.g_fwd is None:
            try:
                self.eng = self._engine(grad_sync)
                self.static = {k: (None if v is None else v.clone()) for k, v in ins.items()}
                torch.cuda.synchronize()
                self.pool = torch.cuda.graph_pool_handle()
                self.g_fwd = torch.cuda.CUDAGraph()
                with graph_capture(self.g_fwd, pool=self.pool):
                    self.eng._pack()                       # re-pack from the live parameters inside the graph
                    self.out = self.eng.forward(*(self.static[k] for k in ("x", "t", "y", "planes", "inv_std")))
                self.keep.append(self.eng.tape)
            except Exception as exc:
                # A capture can still be invalidated by activity outside this call: nothing of it has executed, so this step runs
                # the eager launch sequence and the capture is tried again on a later step (three attempts, then the runner
                # stays eager).
                self._capture_failed(exc)
                eng = self._engine(grad_sync)
                return eng.forward(x, t, y, planes, inv_std), ("eager", eng)
        else:
            for k, v in ins.items():
                self._copy_in(self.static[k], v)
        self.g_fwd.replay()
        self.busy = True
        return self.out.clone(), ("graph", _InFlight(self))

    def flat_of(self, handle) -> torch.Tensor:
        """The flat gradient buffer the backward of `handle` is going to write."""
        kind, obj = handle
        return (obj if kind == "eager" else self.eng).flat

    def backward(self, handle, dout: torch.Tensor) -> Dict[str, torch.Tensor]:
        kind, obj = handle
        if kind == "eager":
            return obj.backward(dout)
        if self.g_bwd is None:
            try:
                self.static["dout"] = dout.to(dtype=torch.float32).contiguous().clone()
                torch.cuda.synchronize()
                self.g_bwd = torch.cuda.CUDAGraph()
                with graph_capture(self.g_bwd, pool=self.pool):
                    self.grads = self.eng.backward(self.static["dout"])
                self.keep.append(self.eng.flat)
            except Exception as exc:
                return self._backward_capture_failed(exc, obj, dout)
        else:
            self.static["dout"].copy_(dout)
        self.g_bwd.replay()
        obj.release()
        # the input gradients live in the graph's memory pool and the next replay rewrites them: hand out copies
        return {k: (v.clone() if k in (DX, DPLANES) else v) for k, v in self.grads.items()}
