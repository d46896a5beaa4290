"""CPU-only tests of the host side: module tree / checkpoint ABI, constructor errors, step tables,
the `sbgm` import shim, and the no-CPU-fallback rule."""
import json
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn as nn

from conftest import GOLDEN_DIR
from oracle import score_ref
from oracle.synth import config_for, param_schema, synth_state_dict


def _build(cfg, device="cpu"):
    from sbgm_danra_b200._smoke import build_model
    return build_model(cfg, synth_state_dict(cfg), "bf16x3", device)


@pytest.mark.parametrize("ck", [dict(n_lr=1), dict(n_lr=2, geo=True, seasons=True),
                                dict(n_lr=1, norm="instance", activation="relu", block_layers=(3, 4, 6, 3)),
                                dict(n_lr=1, use_resize_conv=False, activation="gelu", n_heads=8)])
def test_module_tree_has_reference_state_dict_keys(ck):
    cfg = config_for(**ck)
    net = _build(cfg)       # load_state_dict(strict=True) inside
    mine = {k: tuple(v.shape) for k, v in net.state_dict().items()}
    assert mine == dict(param_schema(cfg))


def test_schema_equals_reference_and_param_count():
    with open(os.path.join(GOLDEN_DIR, "reference_schema.json")) as f:
        ref = json.load(f)["fwd_c1_64_cin2"]
    net = _build(config_for(n_lr=1))
    assert {k: list(v.shape) for k, v in net.state_dict().items()} == ref
    assert sum(p.numel() for p in net.parameters()) == 19_062_082     # SURVEY.md section 2.2


def test_constructor_errors_match_reference():
    from sbgm_danra_b200.score_unet import Decoder, DecoderBlock, Encoder, ImageSelfAttention, SinusoidalEmbedding
    with pytest.raises(ValueError):
        SinusoidalEmbedding(7)
    with pytest.raises(ValueError):
        ImageSelfAttention(64, 5)
    with pytest.raises(ValueError):          # 64 % 3 != 0 inside make_attention_layers -> Optuna prunes on it
        Encoder(1, 256, n_heads=3, device="cpu")
    blk = DecoderBlock(64, 32, 256, device="cpu", norm="group", activation=nn.SiLU)
    assert isinstance(blk.norm1, nn.GroupNorm) and blk.norm1.num_groups == 8
    assert isinstance(DecoderBlock(64, 32, 256, device="cpu").norm1, nn.InstanceNorm2d)
    dec = Decoder(512, 1, 256, device="cpu", norm="group", activation=nn.SiLU)
    assert [(b.input_channels, b.output_channels, b.compute_attn) for b in dec.residual_layers] == \
        [(512, 256, True), (256, 128, True), (128, 64, False), (64, 64, False)]
    assert isinstance(dec.final_layer.norm1, nn.Identity) and isinstance(dec.final_layer.activation, nn.Identity)


def test_no_cpu_fallback():
    from sbgm_danra_b200 import score_sampling as ss
    from sbgm_danra_b200.score_unet import diffusion_coeff_fn, marginal_prob_std_fn
    net = _build(config_for(n_lr=1))
    x, t, c = torch.randn(1, 1, 32, 32), torch.rand(1), torch.randn(1, 1, 32, 32)
    with pytest.raises(RuntimeError, match="no CPU"):
        net(x, t, None, c)
    with pytest.raises(RuntimeError, match="CUDA"):
        ss.Euler_Maruyama_sampler(lambda *a: a[0], marginal_prob_std_fn, diffusion_coeff_fn, batch_size=1, num_steps=2,
                                  device="cpu", img_size=32)


def test_sde_scalars_match_reference_golden(golden):
    from sbgm_danra_b200.score_unet import diffusion_coeff_fn, marginal_prob_std_fn
    t = torch.from_numpy(golden["sde/t"])
    np.testing.assert_allclose(marginal_prob_std_fn(t).numpy(), golden["sde/std"], rtol=1e-6)
    np.testing.assert_allclose(diffusion_coeff_fn(t).numpy(), golden["sde/g"], rtol=1e-6)


def test_step_tables_follow_reference_arithmetic():
    from sbgm_danra_b200 import score_sampling as ss
    n, eps = 7, 1e-3
    em = ss._table_em(score_ref.marginal_prob_std, score_ref.diffusion_coeff, n, eps)
    ts = torch.linspace(1.0, eps, n)
    dt = ts[0] - ts[1]
    g = score_ref.diffusion_coeff(ts)
    assert torch.equal(em[:, 0], ts) and torch.equal(em[:, 1], g)
    assert torch.allclose(em[:, 4], g ** 2 * dt, rtol=1e-7) and torch.allclose(em[:, 5], torch.sqrt(dt) * g, rtol=1e-7)
    assert torch.allclose(em[:, 3], 1.0 / score_ref.marginal_prob_std(ts), rtol=1e-7)
    pc = ss._table_pc(score_ref.marginal_prob_std, score_ref.diffusion_coeff, n, eps)
    ts64 = np.linspace(1.0, eps, n)
    assert np.array_equal(pc[:, 0].numpy(), ts64.astype(np.float32))
    gp = score_ref.diffusion_coeff(torch.from_numpy(ts64.astype(np.float32)))
    assert torch.allclose(pc[:, 5], torch.sqrt(gp ** 2 * (ts64[0] - ts64[1])), rtol=1e-7)


def test_cfg_lookup_and_mask_strip():
    from sbgm_danra_b200 import score_sampling as ss
    assert ss._cfg_scale(None, False) is None
    assert ss._cfg_scale({"classifier_free_guidance": {"enabled": True}}, False) == 2.0
    c = {"classifier_free_guidance": {"enabled": True, "guidance_scale": 5.0, "guidance_scale_max": 3.0}}
    assert ss._cfg_scale(c, clamp=True) == 3.0 and ss._cfg_scale(c, clamp=False) == 5.0   # only pc_sampler clamps
    v = torch.ones(2, 2, 4, 4)
    s = ss._strip_mask(v)
    assert s[:, 0].eq(1).all() and s[:, 1].eq(0).all() and v.eq(1).all()
    assert ss._strip_mask(torch.ones(2, 3, 4, 4)).eq(1).all()


def test_import_shim_redirects_reference_imports():
    import sbgm_danra_b200
    saved = {k: sys.modules.get(k) for k in ("sbgm", "sbgm.score_unet", "sbgm.score_sampling")}
    try:
        for k in saved:
            sys.modules.pop(k, None)
        sbgm_danra_b200.install_as_sbgm()
        from sbgm.score_sampling import Euler_Maruyama_sampler, guided_score_fn, ode_sampler, pc_sampler  # noqa: F401
        from sbgm.score_unet import (Decoder, Encoder, ScoreNet, diffusion_coeff_fn, loss_fn,  # noqa: F401
                                     marginal_prob_std_fn)
        from sbgm_danra_b200.score_unet import ScoreNet as Mine
        assert ScoreNet is Mine
    finally:
        for k, v in saved.items():
            sys.modules.pop(k, None)
            if v is not None:
                sys.modules[k] = v


def test_bn_fold_algebra_on_cpu():
    """engine._Packer.conv folds eval-mode BatchNorm exactly (checked with torch on CPU tensors)."""
    import torch.nn.functional as F
    from sbgm_danra_b200 import engine
    g = torch.Generator().manual_seed(0)
    sd = {"c.weight": torch.randn(16, 8, 3, 3, generator=g), "bn.weight": torch.rand(16, generator=g) + 0.5,
          "bn.bias": torch.randn(16, generator=g), "bn.running_mean": torch.randn(16, generator=g),
          "bn.running_var": torch.rand(16, generator=g) + 0.5}
    cw = engine._Packer(sd, engine.FMT_F32, "cpu").conv("c.weight", bn="bn")
    x = torch.randn(2, 8, 6, 6, generator=g)
    w = cw.w.reshape(3, 3, 8, 16).permute(3, 2, 0, 1)
    got = F.conv2d(x, w, cw.bias, padding=1)
    want = F.batch_norm(F.conv2d(x, sd["c.weight"], padding=1), sd["bn.running_mean"], sd["bn.running_var"],
                        sd["bn.weight"], sd["bn.bias"], False, 0.0, 1e-5)
    assert torch.allclose(got, want, atol=1e-5)
    hi_lo = engine._split_bf16(x)
    assert (hi_lo[0].float() + hi_lo[1].float() - x).abs().max() < 2e-5 * x.abs().max()


def test_gradients_aliasing_the_flat_buffer_are_detached_before_it_is_rewritten():
    """score_unet._detach_grads_aliasing: a `.grad` that is a view of the engine's flat gradient buffer gets its own storage
    (values kept) before the buffer is overwritten; independent gradients and missing gradients are left alone."""
    from sbgm_danra_b200.score_unet import _detach_grads_aliasing
    flat = torch.arange(12, dtype=torch.float32)
    a, b, c = (nn.Parameter(torch.zeros(2, 3)), nn.Parameter(torch.zeros(6)), nn.Parameter(torch.zeros(4)))
    a.grad = flat[0:6].view(2, 3)
    own = torch.full((6,), 7.0)
    b.grad = own
    _detach_grads_aliasing((a, b, c), flat)
    flat.zero_()                                   # what the next captured forward does
    assert torch.equal(a.grad, torch.arange(6, dtype=torch.float32).view(2, 3))
    assert a.grad.untyped_storage().data_ptr() != flat.untyped_storage().data_ptr()
    assert b.grad is own and c.grad is None
    _detach_grads_aliasing((a, b, c), None)        # no captured engine yet: nothing to do


def test_deepcopy_and_pickle_leave_device_caches_behind():
    """`copy.deepcopy(model)` (the reference's EMA copy, sbgm/training.py:114) and whole-model pickles carry parameters and
    buffers, not the derived device state (packed weights, captured graphs), which is neither copyable nor shareable."""
    import copy
    import pickle
    import threading
    net = _build(config_for(n_lr=1))
    net.precision = "bf16"
    net._cache.key, net._cache.value = "k", threading.Lock()            # stand-ins for engines / CUDA graphs
    net.__dict__["_train_runners"] = {"cfg": threading.Lock()}
    net._grad_sync = threading.Lock()
    for twin in (copy.deepcopy(net), pickle.loads(pickle.dumps(net))):
        assert twin._cache is not net._cache and twin._cache.key is None and twin._cache.value is None
        assert "_train_runners" not in twin.__dict__
        assert getattr(twin, "_grad_sync", None) is None and twin.precision == "bf16"
        assert twin.debug_pre_sigma_div == net.debug_pre_sigma_div and twin.training == net.training
        a, b = net.state_dict(), twin.state_dict()
        assert list(a) == list(b)
        assert all(torch.equal(a[k], b[k]) and a[k].data_ptr() != b[k].data_ptr() for k in a)
    assert net.__dict__["_train_runners"] and net._cache.key == "k"      # the original keeps its own


@pytest.mark.parametrize("tol", [1e-5, 1e-3])
def test_resident_rk45_follows_scipy_step_for_step(tol):
    """`score_sampling._rk45_resident` (the opt-in device-resident integrator of ode_sampler) against the integrator the
    reference calls, `scipy.integrate.solve_ivp(method='RK45')` (sbgm/score_sampling.py:296), on the probability-flow ODE of
    a Gaussian-mixture-like analytic score, integrated backwards from t=1 to eps as the sampler does: same number of
    right-hand-side evaluations (= same accepted / rejected step sequence) and the same end state to float64 round-off."""
    from scipy import integrate
    from sbgm_danra_b200.score_sampling import _rk45_resident
    n, sigma, eps = 4096, 25.0, 1e-3
    g = torch.Generator().manual_seed(3)
    mu = torch.randn(n, generator=g, dtype=torch.float64)
    var1 = (sigma ** 2 - 1.0) / (2.0 * np.log(sigma))
    y0 = torch.randn(n, generator=g, dtype=torch.float64) * np.sqrt(var1)

    def rhs_np(t, y):
        var = (sigma ** (2 * t) - 1.0) / (2.0 * np.log(sigma))
        score = -(y - mu.numpy() * np.tanh(y)) / (1.0 + var)
        return -0.5 * sigma ** (2 * t) * score

    def rhs_t(t, y):
        var = (sigma ** (2 * t) - 1.0) / (2.0 * np.log(sigma))
        score = -(y - mu * torch.tanh(y)) / (1.0 + var)
        return -0.5 * sigma ** (2 * t) * score

    res = integrate.solve_ivp(rhs_np, (1.0, eps), y0.numpy(), rtol=tol, atol=tol, method="RK45")
    got, nfev = _rk45_resident(rhs_t, 1.0, eps, y0, tol, tol)
    assert res.status == 0 and nfev == res.nfev, (nfev, res.nfev)
    want = torch.from_numpy(res.y[:, -1])
    assert got.dtype == torch.float64 and float((got - want).abs().max() / want.abs().max()) < 1e-11


def test_resident_rk45_edge_cases():
    from sbgm_danra_b200.score_sampling import _rk45_resident
    y0 = torch.ones(8, dtype=torch.float64)
    out, nfev = _rk45_resident(lambda t, y: -y, 0.5, 0.5, y0, 1e-6, 1e-6)          # empty interval
    assert torch.equal(out, y0) and nfev == 1
    out, nfev = _rk45_resident(lambda t, y: torch.zeros_like(y), 1.0, 0.0, y0, 1e-6, 1e-6)   # zero field: error norm 0 path
    assert torch.equal(out, y0)
    out, _ = _rk45_resident(lambda t, y: -y, 0.0, 1.0, y0, 1e-8, 1e-8)            # forward direction
    assert float((out - np.exp(-1.0)).abs().max()) < 1e-7


def test_flat_gradient_buffer_is_in_forward_order():
    """parallel.GradBucketer launches buckets from the END of the flat buffer as backward fills them: the buffer must be in
    forward order, with the time projections / label embedding (produced by backward's very last launch) at the start."""
    from sbgm_danra_b200.synth import config_for, param_schema
    from sbgm_danra_b200.train_engine import flat_order
    cfg = config_for(n_lr=2, geo=True, seasons=True)
    names = [k for k in param_schema(cfg) if not k.endswith(("running_mean", "running_var", "num_batches_tracked", ".W"))]
    order = flat_order(names)
    assert sorted(order) == sorted(names)
    pos = {k: i for i, k in enumerate(order)}
    first = lambda prefix: min(i for k, i in pos.items() if k.startswith(prefix) and "time_projection" not in k)
    last = lambda prefix: max(i for k, i in pos.items() if k.startswith(prefix) and "time_projection" not in k)
    chain = ["encoder.conv1.", "encoder.conv2.", "encoder.layer1.", "encoder.layer2.", "encoder.layer3.", "encoder.attention_layers.3.",
             "encoder.layer4.", "encoder.attention_layers.4.", "decoder.residual_layers.0.", "decoder.residual_layers.1.",
             "decoder.residual_layers.2.", "decoder.residual_layers.3.", "decoder.final_layer."]
    for a, b in zip(chain, chain[1:]):
        assert last(a) < first(b), (a, b)
    tail = [k for k in names if "time_projection_layer" in k or k.endswith("label_emb.weight")]
    assert tail and max(pos[k] for k in tail) < first("encoder.conv1.")
    # the projection weights, then the biases, each one contiguous run in head order (encoder 0..4, decoder blocks, then the
    # final layer's unused one): TrainEngine.backward lets the time-embedding kernel write the nine used ones in place
    tw = [k for k in order if "time_projection_layer" in k and k.endswith(".weight")]
    tb = [k for k in order if "time_projection_layer" in k and k.endswith(".bias")]
    assert len(tw) == len(tb) == 10 and tw[-1].startswith("decoder.final_layer.")
    assert [pos[k] for k in tw] == list(range(pos[tw[0]], pos[tw[0]] + 10)) and [pos[k] for k in tb] == list(range(pos[tb[0]], pos[tb[0]] + 10))
    assert pos[tw[-1]] < pos[tb[0]] and [k.replace(".weight", "") for k in tw] == [k.replace(".bias", "") for k in tb]


def test_bucketer_gives_the_last_produced_gradients_their_own_first_bucket():
    """The gradients that backward's final kernels produce together (time projections, label embedding) must not share a bucket
    with gradients that are ready earlier: that bucket could only be exchanged after backward (measured: 75 us exposed)."""
    from sbgm_danra_b200.parallel import GradBucketer
    from sbgm_danra_b200.synth import config_for, param_schema
    from sbgm_danra_b200.train_engine import flat_order
    cfg = config_for(n_lr=2, geo=True, seasons=True)
    schema = param_schema(cfg)
    names = flat_order([k for k in schema if not k.endswith(("running_mean", "running_var", "num_batches_tracked", ".W"))])
    layout, off = [], 0
    for k in names:
        n = 1
        for d in schema[k]:
            n *= d
        layout.append((k, off, n))
        off += (n + 63) // 64 * 64
    b = GradBucketer(layout, off, bucket_elems=(32 << 20) // 4, expected=names)
    late = [k for k in names if "time_projection_layer" in k or k.endswith("label_emb.weight")]
    first_bucket = {k for k in names if b.bucket_of[k] == 0}
    assert first_bucket == set(late)
    assert b.bounds[0][1] == max(o + (n + 63) // 64 * 64 for k, o, n in layout if k in first_bucket)
    # backward order: everything else first (decoder ... stem), the late group at the very end -> only bucket 0 is left for the end
    fired = []
    for k in reversed([k for k in names if k not in first_bucket]):
        fired += b.touch([k])
    assert sorted(fired) == list(range(1, len(b.bounds)))
    assert b.touch(late) == [0]


def test_broadcast_style_write_invalidates_engine_cache_key():
    """parallel.broadcast_parameters writes through t.detach() (shares the version counter) so that score_unet._EngineCache
    sees the update; a write through t.data would not bump the version."""
    import torch
    from sbgm_danra_b200.score_unet import _versions
    lin = torch.nn.Linear(3, 2)
    v0 = _versions(lin)
    with torch.no_grad():
        lin.weight.detach().copy_(torch.ones(2, 3))
    assert _versions(lin) != v0
    v1 = _versions(lin)
    lin.weight.data.copy_(torch.zeros(2, 3))          # the pattern the cache cannot see (documented in INTEGRATION.md)
    assert _versions(lin) == v1


def test_graph_capture_pauses_the_cyclic_collector_and_restores_it(monkeypatch):
    """`_capture.graph_capture` collects before the capture, keeps the cyclic collector off inside it (a dead cycle owning a CUDA
    graph must not be finalised mid-capture), asks for thread-local error mode and restores the collector -- also when the body
    raises, and without switching it on for a caller that had it off."""
    import contextlib
    import gc
    from sbgm_danra_b200 import _capture
    seen = {}

    @contextlib.contextmanager
    def fake_graph(graph, **kw):
        seen.update(kw, graph=graph, gc_inside=gc.isenabled())
        yield

    monkeypatch.setattr(torch.cuda, "graph", fake_graph)
    collected = []
    monkeypatch.setattr(_capture.gc, "collect", lambda *a: collected.append(1) or 0)
    assert gc.isenabled()
    with _capture.graph_capture("g", pool="p"):
        assert not gc.isenabled()
    assert gc.isenabled() and collected == [1]
    assert seen == dict(graph="g", pool="p", capture_error_mode="thread_local", gc_inside=False)
    with pytest.raises(RuntimeError):
        with _capture.graph_capture("g"):
            raise RuntimeError("capture invalidated")
    assert gc.isenabled()
    gc.disable()
    try:
        with _capture.graph_capture("g"):
            pass
        assert not gc.isenabled()
    finally:
        gc.enable()


class _FakeTrainEngine:
    """Stands in for train_engine.TrainEngine in the runner's state-machine test: forward = 2x, backward = {"w": 3 dout}."""
    made = 0

    def __init__(self):
        type(self).made += 1
        self.grad_sync, self.tape, self.flat = None, object(), torch.zeros(4)
        self.tk = type("TK", (), {})()
        self.forwards = self.backwards = 0

    def _pack(self):
        pass

    def forward(self, x, t, y, planes, inv_std):
        self.forwards += 1
        return 2 * x

    def backward(self, dout):
        self.backwards += 1
        return {"w": 3 * dout}


def _fake_cuda_graphs(monkeypatch, fail):
    """CUDA-graph stand-ins on CPU: the capture context runs its body once (or raises when `fail` pops True), replay is a no-op."""
    import contextlib
    from sbgm_danra_b200 import train_engine

    class FakeGraph:
        def replay(self):
            pass

    @contextlib.contextmanager
    def fake_capture(graph, **kw):
        if fail and fail.pop(0):
            raise RuntimeError("operation failed due to a previous error during capture")
        yield

    monkeypatch.setattr(train_engine, "graph_capture", fake_capture)
    monkeypatch.setattr(torch.cuda, "CUDAGraph", FakeGraph)
    monkeypatch.setattr(torch.cuda, "graph_pool_handle", lambda: (0, 0))
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a: None)
    return train_engine


def _runner_step(runner, x, sync=None):
    out, handle = runner.forward(x, None, None, None, None, sync)
    grads = runner.backward(handle, torch.ones_like(x))
    return out, grads, handle[0]


def test_train_runner_state_machine_and_capture_failures(monkeypatch):
    """TrainRunner on stand-in graphs: two eager warm-up steps, then capture + replay; a failed forward capture costs one eager
    step and is retried, three failures switch the runner to eager for good; a failed backward capture redoes the step eagerly,
    frees both graphs and leaves the runner idle -- and raises when a gradient exchange over more than one rank is attached."""
    import warnings
    x = torch.arange(4.0)
    fail = [False, False]                                  # first capture pair succeeds
    te = _fake_cuda_graphs(monkeypatch, fail)
    runner = te.TrainRunner(_FakeTrainEngine)
    kinds = [_runner_step(runner, x)[2] for _ in range(4)]
    assert kinds == ["eager", "eager", "graph", "graph"] and runner.g_fwd is not None and runner.g_bwd is not None and not runner.busy
    out, grads, _ = _runner_step(runner, x)
    assert torch.equal(out, 2 * x) and torch.equal(grads["w"], 3 * torch.ones(4))
    # a second forward while a captured step is in flight runs on its own eager engine
    _, h1 = runner.forward(x, None, None, None, None, None)
    _, h2 = runner.forward(x, None, None, None, None, None)
    assert (h1[0], h2[0]) == ("graph", "eager") and runner.busy
    runner.backward(h2, torch.ones(4))
    runner.backward(h1, torch.ones(4))
    assert not runner.busy

    fail[:] = [True, False, False]                         # forward capture fails once, then the pair succeeds
    runner = te.TrainRunner(_FakeTrainEngine)
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always")
        kinds = [_runner_step(runner, x)[2] for _ in range(5)]
    assert kinds == ["eager", "eager", "eager", "graph", "graph"] and runner.capture_failures == 1 and runner.use_graphs
    assert any("capture will be retried" in str(w.message) for w in caught)

    fail[:] = [True, True, True]
    runner = te.TrainRunner(_FakeTrainEngine)
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always")
        kinds = [_runner_step(runner, x)[2] for _ in range(7)]
    assert kinds == ["eager"] * 7 and runner.capture_failures == 3 and not runner.use_graphs and fail == []
    assert any("staying on the eager launch sequence" in str(w.message) for w in caught)

    fail[:] = [False, True, False, False]                  # forward capture fine, backward capture fails, next step captures both
    runner = te.TrainRunner(_FakeTrainEngine)
    with warnings.catch_warnings(record=True):
        warnings.simplefilter("always")
        res = [_runner_step(runner, x) for _ in range(5)]
    assert [r[2] for r in res] == ["eager", "eager", "graph", "graph", "graph"] and runner.capture_failures == 1
    assert all(torch.equal(r[0], 2 * x) and torch.equal(r[1]["w"], 3 * torch.ones(4)) for r in res)
    assert runner.g_fwd is not None and runner.g_bwd is not None and not runner.busy and fail == []

    class Sync:
        world, sync_bn, group = 2, False, None

    fail[:] = [False, True]
    runner = te.TrainRunner(_FakeTrainEngine)
    with warnings.catch_warnings(record=True):
        warnings.simplefilter("always")
        _runner_step(runner, x, Sync())
        _runner_step(runner, x, Sync())
        with pytest.raises(RuntimeError, match="data-parallel"):
            _runner_step(runner, x, Sync())
    assert runner.g_fwd is None and runner.g_bwd is None and not runner.busy
