"""Drop-in mirror of the reference's `sbgm/score_sampling.py`: VE-SDE samplers on sm_100a kernels.

`Euler_Maruyama_sampler`, `pc_sampler`, `ode_sampler`, `guided_score_fn` keep the reference's
signatures (score_sampling.py:63-127, :136-230, :239-300, :10-56).  When `score_model` is this
package's `ScoreNet` the whole sampler step -- time projections, UNet forward, 1/std scaling,
drift + diffusion update with in-kernel Philox noise (and the Langevin corrector for PC) -- is
captured once in a CUDA graph and replayed `num_steps` times; the step index lives on the device.

Differences from the reference, all deliberate (SURVEY.md section 0):
  * EM/ODE initial state honours `img_size` (the reference hard-codes 32 and crashes otherwise);
  * noise comes from a counter-based Philox stream keyed by (seed, global member index, draw), not
    from torch's global generator: `manual_seed()` below controls it, and an ensemble sharded over
    several GPUs (`set_ensemble_shard`) reproduces the single-GPU stream member by member;
  * `ode_sampler` forwards the conditioning tensors to the model (the reference drops them).
"""
from __future__ import annotations

import logging
import os
from dataclasses import dataclass
from typing import Callable, Optional

import numpy as np
import torch

from . import engine as _eng
from ._capture import graph_capture
from ._lib import STEP_COLS, call
from ._lib import stats as _lib_stats

logger = logging.getLogger(__name__)

CFG_WIDE_BELOW = 16        # classifier-free guidance as one 2B-wide evaluation below this many members
num_steps = 800
signal_to_noise_ratio = 0.16
error_tolerance = 1e-5


# ---- noise stream / sharding state ------------------------------------------------------------
@dataclass
class _NoiseState:
    seed: int = 0x5B6D0DA1
    calls: int = 0
    first_member: int = 0          # index of this rank's first member in the global ensemble
    members_total: Optional[int] = None
    group: object = None           # torch.distributed process group for the PC grad-norm exchange


_state = _NoiseState()


def manual_seed(seed: int) -> None:
    """Seed the Philox noise stream; the next sampler / loss call uses exactly `seed`, the one after seed+1, ..."""
    _state.seed, _state.calls = int(seed) & 0xFFFFFFFFFFFFFFFF, 0


def set_ensemble_shard(first_member: int = 0, members_total: Optional[int] = None, group=None) -> None:
    """Declare that this process samples members [first_member, first_member + batch_size) of a
    `members_total`-member ensemble.  EM needs no communication; PC all-gathers one float per member
    per step over `group` so the batch-mean gradient norm (score_sampling.py:201) matches the
    unsharded run exactly."""
    _state.first_member, _state.members_total, _state.group = int(first_member), members_total, group


def noise_state() -> _NoiseState:
    return _state


def _next_seed() -> int:
    s = (_state.seed + _state.calls) & 0xFFFFFFFFFFFFFFFF
    _state.calls += 1
    return s


def _is_native(score_model) -> bool:
    """The fused, graph-captured step serves a ScoreNet of this package: in eval mode on the inference engine (`_NativeStep`),
    in `.train()` -- the reference's generation quirk: `self.model.eval` without parentheses leaves BatchNorm on batch
    statistics while sampling (evaluate_sbgm/generation.py:47) -- on the training engine's forward (`_TrainModeStep`), with
    the batch statistics, the running-statistics updates and, for a sharded ensemble, their all-gather inside the captured step."""
    from .score_unet import ScoreNet
    return isinstance(score_model, ScoreNet)


def _cfg_scale(cfg, clamp: bool) -> Optional[float]:
    """classifier_free_guidance lookup (score_sampling.py:106-110, :180-186)."""
    cfg = cfg or {}
    g = cfg.get("classifier_free_guidance", {})
    if not g.get("enabled", False):
        return None
    scale = g.get("guidance_scale", 2.0)
    if clamp:
        mx = g.get("guidance_scale_max", None)
        if mx is not None and scale > mx:
            scale = mx
    return float(scale)


def _strip_mask(v):
    if v is None or v.shape[1] != 2:
        return v
    v = v.clone()
    v[:, 1] = 0.0
    return v


def guided_score_fn(score_model, x, t, y=None, cond_img=None, lsm_cond=None, topo_cond=None,
                    null_token: int = 0, scale: float = 2.0):
    """Classifier-free guidance: (1 + w) s(x|c) - w s(x|null) with null = zero LR image, geo mask
    channel zeroed, label -> null token (score_sampling.py:10-56)."""
    s_c = score_model(x, t, y, cond_img, lsm_cond, topo_cond)
    s_u = score_model(x, t,
                      torch.full_like(y, null_token) if y is not None else None,
                      torch.zeros_like(cond_img) if cond_img is not None else None,
                      _strip_mask(lsm_cond), _strip_mask(topo_cond))
    if not s_c.is_cuda:
        raise RuntimeError("guided_score_fn: scores must live on a CUDA device (no CPU path)")
    s_c, s_u = s_c.contiguous().float(), s_u.contiguous().float()
    out = torch.empty_like(s_c)
    with torch.cuda.device(s_c.device):
        call("sbgm_cfg_combine", s_c.data_ptr(), s_u.data_ptr(), float(scale), out.data_ptr(), out.numel(), _eng._stream())
    return out


# ---- step tables (host arithmetic identical to the reference's) -------------------------------
def _table_em(marginal_prob_std, diffusion_coeff, n_steps: int, eps: float) -> torch.Tensor:
    ts = torch.linspace(1.0, eps, n_steps)                       # score_sampling.py:96
    dt = ts[0] - ts[1] if n_steps > 1 else torch.tensor(0.0)     # :97
    g = diffusion_coeff(ts).float()                              # :103
    std = marginal_prob_std(ts).float()
    tab = torch.zeros(n_steps, STEP_COLS)
    tab[:, 0], tab[:, 1], tab[:, 2], tab[:, 3] = ts, g, dt, 1.0 / std
    tab[:, 4] = (g ** 2) * dt                                    # :124
    tab[:, 5] = torch.sqrt(dt) * g                               # :125
    return tab


def _table_pc(marginal_prob_std, diffusion_coeff, n_steps: int, eps: float) -> torch.Tensor:
    ts64 = np.linspace(1.0, eps, n_steps)                        # :169 (float64 on the host)
    dt = ts64[0] - ts64[1] if n_steps > 1 else 0.0               # :170
    ts = torch.stack([(torch.ones(1) * tk)[0] for tk in ts64])  # ones(B) * time_step -> fp32, :176
    g = diffusion_coeff(ts).float()                              # :207
    std = marginal_prob_std(ts).float()
    tab = torch.zeros(n_steps, STEP_COLS)
    tab[:, 0], tab[:, 1], tab[:, 2], tab[:, 3] = ts, g, float(dt), 1.0 / std
    tab[:, 4] = (g ** 2) * dt                                    # :224
    tab[:, 5] = torch.sqrt(g ** 2 * dt)                          # :227
    return tab


def _seed_words(seed: int):
    lo, hi = seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF
    return [0, 0, lo - (1 << 32) if lo >= (1 << 31) else lo, hi - (1 << 32) if hi >= (1 << 31) else hi]


class _NativeStep:
    """One fused sampler step on the engine, written so it can be captured in a CUDA graph.  All buffers have
    fixed addresses; a new sampler call with the same shapes only rewrites their contents."""

    def __init__(self, model, batch: int, size: int, n_steps: int, has_y: bool, planes_batch: int, cfg_scale: Optional[float]):
        eng = model.engine()
        self.eng, self.dev, self.b, self.size = eng, eng.device, batch, size
        dev = self.dev
        self.table = torch.zeros((n_steps, STEP_COLS), dtype=torch.float32, device=dev)
        self.counter = torch.zeros(4, dtype=torch.int32, device=dev)       # step, scratch, seed lo, seed hi
        self.inv_std = _eng.InvStd(self.table[:, 3], 0, STEP_COLS, self.counter)
        self.x = torch.zeros((batch, 1, size, size), dtype=torch.float32, device=dev)
        self.score = torch.empty_like(self.x)
        self.mean = torch.empty_like(self.x)
        self.y = torch.zeros(batch, dtype=torch.int64, device=dev) if has_y else None
        if has_y:
            self.tproj_all = None
            self.tproj = torch.empty((batch, eng.tp.c_total), dtype=torch.float32, device=dev)
        else:
            # without labels every member shares the step's time: the projections of ALL steps are computed once per call
            # (load) and a step only selects its row, broadcast over the batch with a zero row stride
            self.tproj_all = torch.empty((n_steps, eng.tp.c_total), dtype=torch.float32, device=dev)
            self.tproj_row = torch.empty((1, eng.tp.c_total), dtype=torch.float32, device=dev)
            self.tproj = self.tproj_row.expand(batch, eng.tp.c_total)
        self.cfg_scale = cfg_scale
        cc = eng.enc.cin - 1
        self.partial = eng.enc.alloc_partial(planes_batch, size, size) if cc > 0 else None
        # classifier-free guidance: the conditional and the null branch as ONE evaluation of 2B members while the GPU is not
        # yet full (score_sampling.py:10-56 runs two B-wide forwards; below ~16 members a forward is launch/latency-bound and
        # the 2B-wide one costs about the same as one B-wide).  SBGM_B200_CFG_WIDE=0: always two evaluations.
        self.wide = cfg_scale is not None and batch < CFG_WIDE_BELOW and os.environ.get("SBGM_B200_CFG_WIDE", "1") != "0"
        if cfg_scale is not None:
            self.partial_u = None if self.partial is None else eng.enc.alloc_partial(planes_batch, size, size)
            self.y_u = None if self.y is None else torch.zeros_like(self.y)
            self.score_c = torch.empty_like(self.x)
            self.score_u = torch.empty_like(self.x)
            self.tproj_u = torch.empty((batch, eng.tp.c_total), dtype=torch.float32, device=dev) if has_y else self.tproj
        if self.wide:
            self.x2 = torch.zeros((2 * batch, 1, size, size), dtype=torch.float32, device=dev)
            self.score2 = torch.empty_like(self.x2)
            self.partial2 = eng.enc.alloc_partial(2 * batch, size, size) if cc > 0 else None      # per member: [cond x B ; null x B]
            self.y2 = torch.zeros(2 * batch, dtype=torch.int64, device=dev) if has_y else None
            self.tproj2 = (torch.empty((2 * batch, eng.tp.c_total), dtype=torch.float32, device=dev) if has_y
                           else self.tproj_row.expand(2 * batch, eng.tp.c_total))
        self.graph = None
        self.per_replay = 0

    @staticmethod
    def planes_of(eng, batch, cond_img, lsm_cond, topo_cond):
        planes = _eng.concat_planes(batch, lsm_cond, topo_cond, cond_img, eng.device)
        cc = eng.enc.cin - 1
        if planes is None:
            if cc != 0:
                raise ValueError(f"model expects {cc} conditioning channels but none were given")
            return None
        if planes.shape[1] != cc:
            raise ValueError(f"model expects {cc} conditioning channels, got {planes.shape[1]}")
        if planes.shape[0] not in (1, batch):
            raise ValueError(f"Batch mismatch: batch_size={batch}, conditions={planes.shape[0]}.")
        if planes.shape[0] > 1 and bool((planes == planes[:1]).all()):
            planes = planes[:1].contiguous()     # every member shares one conditioning sample: broadcast
        return planes

    def load(self, table: torch.Tensor, seed: int, y, planes, planes_u) -> None:
        """Rewrite the call-specific contents (step table, seed, labels, conditioning partial sums) in place."""
        self.table.copy_(table)
        self.counter.copy_(torch.tensor(_seed_words(seed), dtype=torch.int32))
        if self.tproj_all is not None:
            self.eng.tp(self.table, None, rows=self.table.shape[0], t_row_stride=STEP_COLS, t_step_stride=0, out=self.tproj_all)
        if self.y is not None:
            self.y.copy_(y.to(device=self.dev, dtype=torch.int64).reshape(-1))
        self._load_planes(planes, planes_u)
        if self.wide:
            if self.y2 is not None:
                self.y2[:self.b].copy_(self.y)
                self.y2[self.b:].zero_()                              # null token
            if self.partial2 is not None:
                for half, src in enumerate((self.partial, self.partial_u)):
                    dst_t = self.partial2 if isinstance(self.partial2, torch.Tensor) else self.partial2.buf
                    src_t = src if isinstance(src, torch.Tensor) else src.buf
                    nd = dst_t.dim() - 4                              # leading plane dimension of the split-bf16 format
                    dsl = (slice(None),) * nd + (slice(half * self.b, (half + 1) * self.b),)
                    shape = tuple(dst_t.shape[:nd]) + (self.b,) + tuple(dst_t.shape[nd + 1:])
                    dst_t[dsl].copy_(src_t.expand(shape) if src_t.shape[nd] == 1 else src_t)

    def _load_planes(self, planes, planes_u) -> None:
        """The stem's step-invariant contribution of the conditioning planes (and of the null branch's)."""
        if self.partial is not None:
            self.eng.enc.stem_partial(planes, self.size, self.size, out=self.partial)
            if self.cfg_scale is not None:
                self.eng.enc.stem_partial(planes_u, self.size, self.size, out=self.partial_u)

    def _forward(self, partial, y, tproj, out, x=None) -> None:
        x = self.x if x is None else x
        if self.tproj_all is not None:
            call("sbgm_select_step_row", self.tproj_all.data_ptr(), self.tproj_all.shape[1], self.counter.data_ptr(),
                 self.tproj_row.data_ptr(), _eng._stream())
        else:
            self.eng.tp(self.table, y, rows=x.shape[0], t_row_stride=0, t_step_stride=STEP_COLS, step_counter=self.counter, out=tproj)
        self._evaluate(x, partial, y, tproj, out)

    def _evaluate(self, x, partial, y, tproj, out) -> None:
        """The network at the step's time projections `tproj` into `out`; `partial`: the conditioning as `_load_planes` left it."""
        fmaps = self.eng.enc.forward(x, None, tproj, partial=partial)
        self.eng.dec.forward(fmaps, tproj, self.inv_std, dst=out)

    def score_into(self, scale: Optional[float] = None) -> torch.Tensor:
        """`scale`: guidance scale of THIS evaluation (the PC corrector clamps it to guidance_scale_max, the predictor does
        not: score_sampling.py:182-186 vs :209-219); default = the plan's scale."""
        if self.cfg_scale is None:
            self._forward(self.partial, self.y, self.tproj, self.score)
        elif self.wide:
            self.x2[:self.b].copy_(self.x)
            self.x2[self.b:].copy_(self.x)
            self._forward(self.partial2, self.y2, self.tproj2, self.score2, x=self.x2)
            call("sbgm_cfg_combine", self.score2[:self.b].data_ptr(), self.score2[self.b:].data_ptr(),
                 self.cfg_scale if scale is None else scale, self.score.data_ptr(), self.score.numel(), _eng._stream())
        else:
            self._forward(self.partial, self.y, self.tproj, self.score_c)
            self._forward(self.partial_u, self.y_u, self.tproj_u, self.score_u)
            call("sbgm_cfg_combine", self.score_c.data_ptr(), self.score_u.data_ptr(), self.cfg_scale if scale is None else scale,
                 self.score.data_ptr(), self.score.numel(), _eng._stream())
        return self.score


class _TrainModeStep(_NativeStep):
    """A sampler step of a ScoreNet left in `.train()` (evaluate_sbgm/generation.py:47): every network evaluation normalises
    with the statistics of the CURRENT batch of members (the ensemble members are coupled) and moves the running statistics
    (momentum 0.1, unbiased variance) and `num_batches_tracked`, exactly as torch's BatchNorm2d does under `no_grad`.  The
    evaluation is `TrainEngine.forward` in sampler mode (step-table time projections and 1/std, no tape, no gradient buffer),
    so the whole step still captures into ONE CUDA graph.  With `set_ensemble_shard(..., group=g)` and fewer local members than
    the ensemble has, the per-channel partial sums are all-gathered over `g` inside the graph (synchronised BatchNorm): R ranks
    x B/R members reproduce the single-process statistics of all B members.  Classifier-free guidance keeps the reference's
    two separate evaluations (each with its own batch statistics): never the 2B-wide form."""

    def __init__(self, model, batch: int, size: int, n_steps: int, has_y: bool, planes, planes_u, cfg_scale: Optional[float],
                 sync_group=None):
        super().__init__(model, batch, size, n_steps, has_y, 0, cfg_scale)
        from .train_engine import TrainEngine
        tensors = dict(model.named_parameters())
        tensors.update(model.named_buffers())
        self.train_eng = TrainEngine(tensors, model.spec(), model.precision, self.dev, bn_train=True)
        self.train_eng.tk.sync_bn = sync_group
        self.bn_counters = [m.num_batches_tracked for m in model._bn_modules()]
        self.wide = False
        # conditioning planes as static buffers (the training engine's stem reads them every evaluation)
        self.partial = None if planes is None else torch.empty_like(planes)
        self.partial_u = None if planes_u is None else torch.empty_like(planes_u)

    def _load_planes(self, planes, planes_u) -> None:
        if self.partial is not None:
            self.partial.copy_(planes)
        if self.partial_u is not None:
            self.partial_u.copy_(planes_u)

    def _evaluate(self, x, partial, y, tproj, out) -> None:
        # weights were packed when the plan was built (the plan is keyed on the parameter versions); the running statistics are
        # read and updated live
        self.train_eng.forward(x, None, y, partial, None, sampler=dict(tproj=tproj, inv_std=self.inv_std, dst=out))
        torch._foreach_add_(self.bn_counters, 1)


class _GenericStep:
    """Same update kernels around an arbitrary `score_model` callable (no CUDA graph)."""

    def __init__(self, score_model, batch, size, table, device, y, cond_img, lsm_cond, topo_cond, cfg_scale):
        dev = torch.device(device)
        if dev.type != "cuda":
            raise RuntimeError("samplers run on CUDA devices only (no CPU fallback); got device=" + str(device))
        self.dev, self.b, self.size = dev, batch, size
        self.model, self.args = score_model, (y, cond_img, lsm_cond, topo_cond)
        self.table = table.to(dev).contiguous()
        self.table_host = table
        self.counter = torch.zeros(4, dtype=torch.int32, device=dev)
        self.x = torch.zeros((batch, 1, size, size), dtype=torch.float32, device=dev)
        self.mean = torch.empty_like(self.x)
        self.cfg_scale = cfg_scale
        self.k = 0
        self.graph = None

    def score_into(self, scale: Optional[float] = None) -> torch.Tensor:
        bt = torch.full((self.b,), float(self.table_host[self.k, 0]), dtype=torch.float32, device=self.dev)
        if self.cfg_scale is None:
            s = self.model(self.x, bt, *self.args)
        else:
            s = guided_score_fn(self.model, self.x, bt, *self.args, scale=self.cfg_scale if scale is None else scale)
        self.score = s.contiguous().float()
        return self.score


def _predict(st, draw_base, draw_stride, first_elem) -> None:
    call("sbgm_sampler_predictor", st.x.data_ptr(), st.score.data_ptr(), st.mean.data_ptr(), st.x.numel(),
         st.table.data_ptr(), st.counter.data_ptr(), draw_base, draw_stride, first_elem, _eng._stream())


def _correct(st, sumsq, sumsq_all, snr, first_elem) -> None:
    per = st.size * st.size
    call("sbgm_sampler_sumsq", st.score.data_ptr(), sumsq.data_ptr(), st.b, per, _eng._stream())
    if sumsq_all is not sumsq:
        import torch.distributed as dist
        dist.all_gather_into_tensor(sumsq_all, sumsq, group=_state.group)
    call("sbgm_sampler_corrector", st.x.data_ptr(), st.score.data_ptr(), sumsq_all.data_ptr(), sumsq_all.numel(), per,
         float(snr), st.x.numel(), st.counter.data_ptr(), 1, 2, first_elem, _eng._stream())


# captured sampler plans (buffers + CUDA graph), most recent first; each holds one forward's activations
_PLAN_CACHE: list = []
_PLAN_CACHE_SIZE = 2


def clear_sampler_cache() -> None:
    """Drop the cached CUDA graphs / activation pools of previous sampler calls."""
    _PLAN_CACHE.clear()


def _sample(kind: str, score_model, marginal_prob_std, diffusion_coeff, batch_size, n_steps, snr, device, eps, img_size,
            y, cond_img, lsm_cond, topo_cond, cfg, use_graph: bool = True) -> torch.Tensor:
    if img_size % 32 != 0:
        raise ValueError(f"img_size must be a multiple of 32, got {img_size}")
    seed = _next_seed()
    table = (_table_em if kind == "em" else _table_pc)(marginal_prob_std, diffusion_coeff, n_steps, eps)
    # PC: the corrector's guidance scale is clamped to guidance_scale_max, the predictor re-reads the unclamped one
    # (score_sampling.py:182-186 vs :209-219); EM never clamps (:106-110)
    scale = _cfg_scale(cfg, clamp=False)
    scale_corrector = _cfg_scale(cfg, clamp=True) if kind == "pc" else scale
    native = _is_native(score_model)
    dev = score_model.engine().device if native else torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError("samplers run on CUDA devices only (no CPU fallback); got device=" + str(device))
    per = img_size * img_size
    first_elem = _state.first_member * per
    std1 = float(marginal_prob_std(torch.ones(1))[0])             # score_sampling.py:93-95 / :167-168
    sharded = kind == "pc" and _state.members_total is not None and _state.members_total != batch_size
    total = _state.members_total if sharded else batch_size

    with torch.no_grad(), torch.cuda.device(dev):
        if native:
            eng = score_model.engine()
            planes = _NativeStep.planes_of(eng, batch_size, cond_img, lsm_cond, topo_cond)
            planes_u = None
            if scale is not None and planes is not None:
                planes_u = _NativeStep.planes_of(eng, batch_size, None if cond_img is None else torch.zeros_like(cond_img),
                                                 _strip_mask(lsm_cond), _strip_mask(topo_cond))
                if planes_u.shape[0] != planes.shape[0]:
                    planes_u = planes_u.expand(planes.shape[0], -1, -1, -1).contiguous()
            train_mode = bool(score_model.training)
            # train-mode BatchNorm couples the members: a sharded ensemble synchronises the statistics over the shard group
            bn_group = _state.group if (train_mode and _state.members_total not in (None, batch_size) and _state.group is not None) else None
            # eval: keyed on the packed engine (rebuilt when a parameter changes); train mode: on the model and its parameter
            # versions (the running statistics move every evaluation and must not invalidate the plan)
            owner = ((id(score_model),) + tuple((p_.data_ptr(), p_._version) for p_ in score_model.parameters())) if train_mode else id(eng)
            key = (owner, kind, batch_size, img_size, n_steps, scale, scale_corrector, float(snr), y is not None,
                   0 if planes is None else planes.shape[0], first_elem, total, id(_state.group) if (sharded or bn_group is not None) else 0,
                   use_graph, train_mode)
            st = next((p for k, p in _PLAN_CACHE if k == key), None)
            if st is None:
                # cached across calls and rewritten in place: must be ordinary tensors even when the first caller is inside
                # torch.inference_mode() (inference tensors cannot be updated in place by a later no_grad caller)
                with torch.inference_mode(False):
                    if train_mode:
                        st = _TrainModeStep(score_model, batch_size, img_size, n_steps, y is not None, planes, planes_u, scale, bn_group)
                    else:
                        st = _NativeStep(score_model, batch_size, img_size, n_steps, y is not None,
                                         0 if planes is None else planes.shape[0], scale)
                    st.sumsq = torch.zeros(batch_size, dtype=torch.float32, device=dev)
                    st.sumsq_all = torch.zeros(total, dtype=torch.float32, device=dev) if sharded else st.sumsq
                _PLAN_CACHE.insert(0, (key, st))
                del _PLAN_CACHE[_PLAN_CACHE_SIZE:]
            st.load(table, seed, y, planes, planes_u)
        else:
            st = _GenericStep(score_model, batch_size, img_size, table, dev, y, cond_img, lsm_cond, topo_cond, scale)
            st.counter.copy_(torch.tensor(_seed_words(seed), dtype=torch.int32))
            st.sumsq = torch.zeros(batch_size, dtype=torch.float32, device=dev)
            st.sumsq_all = torch.zeros(total, dtype=torch.float32, device=dev) if sharded else st.sumsq

        def one_step() -> None:
            if kind == "pc":
                st.score_into(scale_corrector)
                _correct(st, st.sumsq, st.sumsq_all, snr, first_elem)
                st.score_into(scale)
                _predict(st, 2, 2, first_elem)
            else:
                st.score_into()
                _predict(st, 1, 1, first_elem)

        if native and use_graph and n_steps > 1 and st.graph is None:
            # eager warm-up step (lazy kernel attributes, scratch buffers), then capture one step
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                one_step()
            torch.cuda.current_stream(dev).wait_stream(side)
            st.graph = torch.cuda.CUDAGraph()
            before = _lib_stats.launches
            with graph_capture(st.graph):
                one_step()
            st.per_replay = _lib_stats.launches - before     # kernels recorded in the graph
            _lib_stats.launches = before
        st.counter[:2].zero_()
        call("sbgm_sampler_init", st.x.data_ptr(), st.x.numel(), std1, seed, first_elem, _eng._stream())
        for k in range(n_steps):
            if st.graph is not None:
                st.graph.replay()
                _lib_stats.launches += st.per_replay
            else:
                if not native:
                    st.k = k
                one_step()
        return st.mean.clone()


def Euler_Maruyama_sampler(score_model, marginal_prob_std, diffusion_coeff, batch_size=64, num_steps=500,
                           device="cuda", eps=1e-3, img_size=64, y=None, cond_img=None, lsm_cond=None,
                           topo_cond=None, cfg=None):
    """Euler-Maruyama reverse-SDE sampler (score_sampling.py:63-127).  Returns the noise-free mean of the last step."""
    return _sample("em", score_model, marginal_prob_std, diffusion_coeff, batch_size, num_steps, 0.0, device, eps,
                   img_size, y, cond_img, lsm_cond, topo_cond, cfg)


def pc_sampler(score_model, marginal_prob_std, diffusion_coeff, batch_size=64, num_steps=num_steps,
               snr=signal_to_noise_ratio, device="cuda", eps=1e-3, img_size=64, y=None, cond_img=None,
               lsm_cond=None, topo_cond=None, cfg=None):
    """Predictor-corrector sampler: Langevin corrector + Euler-Maruyama predictor, 2 NFE per step
    (score_sampling.py:136-230)."""
    return _sample("pc", score_model, marginal_prob_std, diffusion_coeff, batch_size, num_steps, snr, device, eps,
                   img_size, y, cond_img, lsm_cond, topo_cond, cfg)


# Dormand-Prince 5(4) tableau (scipy.integrate.RK45: C, A, B and the error weights E = B5 - B4)
_DP_C = (0.0, 1 / 5, 3 / 10, 4 / 5, 8 / 9, 1.0)
_DP_A = ((), (1 / 5,), (3 / 40, 9 / 40), (44 / 45, -56 / 15, 32 / 9), (19372 / 6561, -25360 / 2187, 64448 / 6561, -212 / 729),
         (9017 / 3168, -355 / 33, 46732 / 5247, 49 / 176, -5103 / 18656))
_DP_B = (35 / 384, 0.0, 500 / 1113, 125 / 192, -2187 / 6784, 11 / 84)
_DP_E = (-71 / 57600, 0.0, 71 / 16695, -71 / 1920, 17253 / 339200, -22 / 525, 1 / 40)


class _TorchStages:
    """Stage arithmetic of `_rk45_resident` with torch float64 ops: what runs when the state is a CPU tensor, i.e. in the
    host-logic tests that pin the CONTROLLER to scipy step for step (tests/test_host_logic.py).  `fun(t, y64) -> f64`."""

    def __init__(self, y0: torch.Tensor, fun) -> None:
        self.fun, self.n = fun, y0.numel()
        self.y = y0.to(torch.float64).reshape(-1).clone()
        self.K = torch.empty((7, self.n), dtype=torch.float64, device=y0.device)
        self.y_new = None

    def _comb(self, coefs, h: float) -> torch.Tensor:
        if not coefs:
            return self.y
        a = torch.tensor(coefs, dtype=torch.float64, device=self.y.device)
        return self.y + torch.mv(self.K[:len(coefs)].T, a) * h

    def eval(self, slot: int, t: float, coefs, h: float) -> None:
        self.K[slot] = self.fun(t, self._comb(coefs, h))

    def propose(self, coefs, h: float, t_new: float) -> None:
        self.y_new = self._comb(coefs, h)
        self.K[6] = self.fun(t_new, self.y_new)

    def sumsq(self, coefs, h: float, atol: float, rtol: float, with_new: bool) -> float:
        a = torch.tensor(coefs, dtype=torch.float64, device=self.y.device)
        v = torch.mv(self.K[:len(coefs)].T, a) * h
        ref = torch.maximum(self.y.abs(), self.y_new.abs()) if with_new else self.y.abs()
        return float(((v / (atol + ref * rtol)) ** 2).sum())

    def sumsq_state(self, atol: float, rtol: float) -> float:
        return float(((self.y / (atol + self.y.abs() * rtol)) ** 2).sum())

    def accept(self) -> None:
        self.y = self.y_new
        self.K[0] = self.K[6]

    def result(self) -> torch.Tensor:
        return self.y


class _KernelStages:
    """The same stage arithmetic on the device (csrc/post_sampler.cu): a stage combination is one launch that also writes
    the float32 copy the network reads, the right-hand side -1/2 g^2 score is scaled into its float64 stage slot by one launch,
    and the scaled error norm is a deterministic two-launch reduction -- one double crosses to the host per attempted step.
    `fun(t, x32) -> (score32, scale)` with x32 / score32 flat float32 tensors of the state's size."""

    def __init__(self, y0: torch.Tensor, fun) -> None:
        from . import _lib
        self.fun, self.n, self.dev = fun, y0.numel(), y0.device
        f64 = dict(dtype=torch.float64, device=self.dev)
        self.y = y0.to(torch.float64).reshape(-1).clone()
        self.y_new = torch.empty(self.n, **f64)
        self.K = torch.empty((7, self.n), **f64)
        self.x32 = torch.empty(self.n, dtype=torch.float32, device=self.dev)
        self.scratch = torch.empty(_lib.query("sbgm_rk45_scratch_doubles", self.n), **f64)
        self.out = torch.empty(1, **f64)

    @staticmethod
    def _row(coefs):
        import ctypes
        return (ctypes.c_double * 7)(*coefs, *([0.0] * (7 - len(coefs))))

    def _rhs(self, slot: int, t: float) -> None:
        score, scale = self.fun(t, self.x32)
        score = score.reshape(-1).contiguous().float()
        call("sbgm_rk45_rhs", score.data_ptr(), float(scale), self.K[slot].data_ptr(), self.n, _eng._stream())

    def eval(self, slot: int, t: float, coefs, h: float) -> None:
        with torch.cuda.device(self.dev):
            call("sbgm_rk45_combine", self.y.data_ptr(), self.K.data_ptr(), self.n, len(coefs), self._row(coefs), float(h), None,
                 self.x32.data_ptr(), _eng._stream())
            self._rhs(slot, t)

    def propose(self, coefs, h: float, t_new: float) -> None:
        with torch.cuda.device(self.dev):
            call("sbgm_rk45_combine", self.y.data_ptr(), self.K.data_ptr(), self.n, len(coefs), self._row(coefs), float(h),
                 self.y_new.data_ptr(), self.x32.data_ptr(), _eng._stream())
            self._rhs(6, t_new)

    def sumsq(self, coefs, h: float, atol: float, rtol: float, with_new: bool) -> float:
        with torch.cuda.device(self.dev):
            call("sbgm_rk45_error_norm", self.K.data_ptr(), self.n, len(coefs), self._row(coefs), float(h), self.y.data_ptr(),
                 self.y_new.data_ptr() if with_new else None, float(atol), float(rtol), self.scratch.data_ptr(), self.out.data_ptr(),
                 _eng._stream())
        return float(self.out.item())

    def sumsq_state(self, atol: float, rtol: float) -> float:
        with torch.cuda.device(self.dev):      # the state itself plays the role of a one-stage "K"
            call("sbgm_rk45_error_norm", self.y.data_ptr(), self.n, 1, self._row([1.0]), 1.0, self.y.data_ptr(), None, float(atol),
                 float(rtol), self.scratch.data_ptr(), self.out.data_ptr(), _eng._stream())
        return float(self.out.item())

    def accept(self) -> None:
        self.y, self.y_new = self.y_new, self.y
        self.K[0].copy_(self.K[6])

    def result(self) -> torch.Tensor:
        return self.y


def _rk45_resident(fun, t0: float, t_bound: float, y0: torch.Tensor, rtol: float, atol: float):
    """Adaptive Dormand-Prince 5(4) with the state, the seven stages and the error estimate resident on `y0`'s device.

    Restates the algorithm of the third-party integrator the reference calls (`integrate.solve_ivp(..., method='RK45')`,
    sbgm/score_sampling.py:296; SciPy 1.18.1: `_ivp/rk.py` rk_step / RungeKutta._step_impl, `_ivp/common.py`
    select_initial_step, norm = RMS): same initial-step rule, error norm, SAFETY 0.9 / MIN_FACTOR 0.2 / MAX_FACTOR 10 step
    control and end-point clipping, so the accepted step sequence is SciPy's up to float64 summation order.  Only the scalar
    error norm crosses to the host (one read per attempted step, it decides accept / reject); SciPy's host version moves
    the whole float64 state across PCIe twice per right-hand side.  On a CUDA state the stage arithmetic runs in this repo's
    kernels (`_KernelStages`; `fun(t, x32) -> (score32, scale)`), on a CPU state in torch (`_TorchStages`; `fun(t, y64) -> f64`,
    the controller's host-logic tests).  Returns (y at t_bound -- or the last accepted state if the step size underflows, which
    is what the reference reads from `res.y[:, -1]` -- and the number of `fun` calls)."""
    import math
    ops = _KernelStages(y0, fun) if y0.is_cuda else _TorchStages(y0, fun)
    n = ops.n
    rtol = max(float(rtol), 100 * np.finfo(float).eps)              # validate_tol
    direction = 1.0 if t_bound >= t0 else -1.0
    nfev = 0
    rms = lambda sumsq: math.sqrt(max(sumsq, 0.0) / n)

    t = float(t0)
    interval = abs(t_bound - t0)
    ops.eval(0, t, (), 0.0)                                          # f = fun(t0, y0)
    nfev += 1
    if n == 0 or interval == 0.0:
        return ops.result(), nfev
    # select_initial_step (norms scaled by atol + |y| rtol)
    d0 = rms(ops.sumsq_state(atol, rtol))
    d1 = rms(ops.sumsq((1.0,), 1.0, atol, rtol, False))
    h0 = 1e-6 if (d0 < 1e-5 or d1 < 1e-5) else 0.01 * d0 / d1
    h0 = min(h0, interval)
    ops.eval(1, t + h0 * direction, (1.0,), h0 * direction)          # f1 = fun(t0 + h0, y0 + h0 f)
    nfev += 1
    d2 = rms(ops.sumsq((-1.0, 1.0), 1.0, atol, rtol, False)) / h0
    h1 = max(1e-6, h0 * 1e-3) if (d1 <= 1e-15 and d2 <= 1e-15) else (0.01 / max(d1, d2)) ** (1 / 5)
    h_abs = min(100 * h0, h1, interval)

    while direction * (t - t_bound) < 0:
        min_step = 10 * abs(float(np.nextafter(t, direction * np.inf)) - t)
        h_abs = max(h_abs, min_step)
        rejected = False
        while True:
            if h_abs < min_step:
                return ops.result(), nfev                            # TOO_SMALL_STEP: the reference reads the last state
            t_new = t + h_abs * direction
            if direction * (t_new - t_bound) > 0:
                t_new = t_bound
            h = t_new - t
            h_abs = abs(h)
            for s in range(1, 6):                                    # rk_step: K[0] holds f(t, y)
                ops.eval(s, t + _DP_C[s] * h, _DP_A[s], h)
            ops.propose(_DP_B, h, t + h)                             # y_new and K[6] = f(t + h, y_new)
            nfev += 6
            err = rms(ops.sumsq(_DP_E, h, atol, rtol, True))
            if err < 1:
                factor = 10.0 if err == 0 else min(10.0, 0.9 * err ** -0.2)
                h_abs *= min(1.0, factor) if rejected else factor
                break
            h_abs *= max(0.2, 0.9 * err ** -0.2)
            rejected = True
        t = t_new
        ops.accept()
    return ops.result(), nfev


def ode_sampler(score_model, marginal_prob_std, diffusion_coeff, num_steps=100, batch_size=64, atol=error_tolerance,
                rtol=error_tolerance, device="cuda", z=None, eps=1e-3, img_size=64, y=None, cond_img=None,
                lsm_cond=None, topo_cond=None, cfg=None):
    """Probability-flow ODE with the adaptive RK45 of `scipy.integrate.solve_ivp` (score_sampling.py:239-300).

    Default: the float64 state, the seven stages and the error estimate stay on the device (`_rk45_resident`: SciPy's
    Dormand-Prince controller restated and pinned to it step for step, stage arithmetic in csrc/post_sampler.cu); one double
    is read back per attempted step.  `SBGM_B200_ODE=host` runs SciPy itself on the host exactly as the reference does, with the
    float64 state crossing PCIe twice per score evaluation (kept as the cross-check: both give the same result to integrator
    round-off, tests/test_gpu_model.py)."""
    from scipy import integrate
    dev = torch.device(device)
    if z is None:
        init = torch.empty((batch_size, 1, img_size, img_size), dtype=torch.float32, device=dev)
        std1 = float(marginal_prob_std(torch.ones(1))[0])
        with torch.cuda.device(dev):
            call("sbgm_sampler_init", init.data_ptr(), init.numel(), std1, _next_seed(),
                 _state.first_member * img_size * img_size, _eng._stream())
    else:
        init = z.to(dev)
    shape = tuple(init.shape)

    def rhs(t, xflat):
        sample = torch.tensor(xflat, device=dev, dtype=torch.float32).reshape(shape)
        ts = torch.full((shape[0],), float(t), device=dev, dtype=torch.float32)
        with torch.no_grad():
            s = score_model(sample, ts, y, cond_img, lsm_cond, topo_cond)
        g = float(diffusion_coeff(torch.tensor(t)))
        return -0.5 * (g ** 2) * s.cpu().numpy().reshape(-1).astype(np.float64)

    if dev.type != "cuda":
        raise RuntimeError("samplers run on CUDA devices only (no CPU fallback); got device=" + str(device))
    if os.environ.get("SBGM_B200_ODE", "resident") != "host":
        def rhs_resident(t, x32):
            ts = torch.full((shape[0],), float(t), device=dev, dtype=torch.float32)
            with torch.no_grad():
                s = score_model(x32.reshape(shape), ts, y, cond_img, lsm_cond, topo_cond)
            g = float(diffusion_coeff(torch.tensor(t)))
            return s, -0.5 * (g ** 2)

        with torch.no_grad():
            out, nfev = _rk45_resident(rhs_resident, 1.0, eps, init.reshape(-1), rtol, atol)
        logger.info(f"Number of function evaluations: {nfev}")
        return out.reshape(shape)
    res = integrate.solve_ivp(rhs, (1.0, eps), init.reshape(-1).cpu().numpy(), rtol=rtol, atol=atol, method="RK45")
    logger.info(f"Number of function evaluations: {res.nfev}")
    return torch.tensor(res.y[:, -1], device=dev).reshape(shape)


def edm_sigma_schedule(n_steps, sigma_min=0.002, sigma_max=80, rho=7.0, device="cuda"):
    """Karras et al. sigma schedule (score_sampling.py:304-306); a host-side helper, unused by the samplers."""
    i = torch.linspace(0, 1, n_steps, device=device)
    return (sigma_max ** (1 / rho) + i * (sigma_min ** (1 / rho) - sigma_max ** (1 / rho))) ** rho


# ---- DSM loss forward (score_unet.py:936-985) --------------------------------------------------
def _dsm_loss_forward(model, x, marginal_prob_std, t_eps, y, cond_img, lsm_cond, topo_cond, sdf_cond):
    from . import _lib
    if not x.is_cuda:
        raise RuntimeError("loss_fn: x must live on a CUDA device (no CPU path)")
    dev = x.device
    seed = _next_seed()
    n, per = x.shape[0], x[0].numel()
    with torch.cuda.device(dev):
        with torch.no_grad():
            x = x.contiguous().float()
            start = _state.first_member // 4 * 4          # Philox counters cover 4 elements: generate from an aligned start
            off = _state.first_member - start
            u = torch.empty((off + n + 3) // 4 * 4, dtype=torch.float32, device=dev)
            call("sbgm_philox_uniform", u.data_ptr(), u.numel(), seed, 0, start, _eng._stream())
            t = u[off:off + n] * (1.0 - t_eps) + t_eps
            std = marginal_prob_std(t).float().contiguous()
            xt, z = torch.empty_like(x), torch.empty_like(x)
            call("sbgm_dsm_perturb", x.data_ptr(), std.data_ptr(), xt.data_ptr(), z.data_ptr(), n, per, seed, 1,
                 _state.first_member * per, _eng._stream())
            sdf = None if sdf_cond is None else sdf_cond.to(dev).contiguous().float()
        score = model(xt, t, y=y, cond_img=cond_img, lsm_cond=lsm_cond, topo_cond=topo_cond)
        from .score_unet import _DSMLossFn
        return _DSMLossFn.apply(score, std, z, sdf)
