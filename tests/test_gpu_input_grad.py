"""GPU: gradients of ScoreNet with respect to its inputs (x and the conditioning planes).

The stem data-gradient kernels are compared with torch.nn.grad.conv2d_input in float64 on the df values they read (the stored
activation format) and the weights they read (bf16: the rounded weight; split bf16: hi + lo); the only error left is fp32
summation order (and, in split bf16, the dropped lo x lo product), so the gates are those of test_gpu_wgrad.py.  The whole network's
vector-Jacobian products torch.autograd.grad(score, inputs, v) are compared with the same call on the CPU oracle in float64.

Some of these products are ill-conditioned: with running-statistics BatchNorm at Cin = 2 the oracle's own float32 result is 8.5e-3
away from its float64 one (at Cin = 7 it is 1.4e-6), so every gate is at least twice the float32 oracle's error.  The split formats
(bf16x3, and fp16x2, which trains on bf16x3) meet the whole-gradient gate of the parameter gradients (1e-3) on most cases but not
all (measured up to 1.1e-2 at Cin = 2 with batch statistics, 2.1e-3 at Cin = 7): their gate is also at most a tenth of the error of
the oracle under bf16 autocast, the yardstick of the bf16 mode (measured: 2e-1)."""
import functools
import os
import shutil
import subprocess

import pytest
import torch

from conftest import rel_l2

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
FMTS = {"fp32": 0, "bf16": 1, "bf16x3": 2}
KERNEL_GATE = {"fp32": 2e-5, "bf16": 1e-5, "bf16x3": 5e-5}
NET_GATE = {"fp32": 1e-4, "bf16x3": 1e-3, "fp16x2": 1e-3}
SPLIT_FRACTION_OF_AUTOCAST = 0.1
PARAM_ONLY = {"sbgm_conv2d_wgrad_tc", "sbgm_conv2d_wgrad_simt", "sbgm_wgrad_reduce", "sbgm_stem_wgrad", "sbgm_channel_sums",
              "sbgm_time_embed_backward"}


def gen(*shape, seed=0):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed))


# ---- 1. the kernels ------------------------------------------------------------------------------------------------------
def run_stem_dgrad(prec, df_act, w1, np_, cc, n, h, w):
    from sbgm_danra_b200 import _lib
    from sbgm_danra_b200._lib import call
    from sbgm_danra_b200.train_engine import PackPlan, stem_dgrad_weight
    fmt = FMTS[prec]
    dx = torch.full((n, 1, h, w), float("nan"), device=DEV)
    dpl = torch.full((np_, cc, h, w), float("nan"), device=DEV) if cc else None
    ws = torch.full((max(_lib.query("sbgm_stem_dgrad_workspace_floats", np_, cc, n, h, w), 1),), float("nan"), device=DEV)
    st = torch.cuda.current_stream().cuda_stream
    if prec == "fp32":
        call("sbgm_stem_dgrad_simt", df_act.ptr, df_act.plane, fmt, w1.data_ptr(), dx.data_ptr(), None if dpl is None else dpl.data_ptr(),
             np_, cc, n, h, w, ws.data_ptr(), st)
    else:
        plan = PackPlan(fmt)
        table = stem_dgrad_weight(plan, w1)
        plan.run()
        call("sbgm_stem_dgrad_tc", df_act.ptr, df_act.plane, fmt, table.data_ptr(), table.stride(1), dx.data_ptr(),
             None if dpl is None else dpl.data_ptr(), np_, cc, n, h, w, ws.data_ptr(), st)
    torch.cuda.synchronize()
    return dx.cpu(), None if dpl is None else dpl.cpu()


def weight_as_read(prec, w1):
    if prec == "bf16":
        return w1.bfloat16().double()
    return w1.double()


@pytest.mark.parametrize("prec", ["fp32", "bf16", "bf16x3"])
@pytest.mark.parametrize("cin", [1, 2, 7, 15])
@pytest.mark.parametrize("shared", [False, True])
@pytest.mark.parametrize("size", [32, 96, 128, 256])
def test_stem_dgrad_kernel_matches_float64(prec, cin, shared, size):
    from sbgm_danra_b200.engine import Act
    n = 3 if size < 256 else 2
    cc = cin - 1
    if shared and cc == 0:
        pytest.skip("no conditioning planes to share")
    np_ = 1 if shared else n
    fmt = FMTS[prec]
    w1 = (gen(64, cin, 8, 8, seed=cin) / 16).to(DEV)
    df = Act.from_nchw(gen(n, 64, size // 2, size // 2, seed=size).to(DEV), fmt)
    df64 = df.to_nchw().cpu().double()
    ref = torch.nn.grad.conv2d_input((n, cin, size, size), weight_as_read(prec, w1.cpu()), df64, stride=2, padding=3)
    dx, dpl = run_stem_dgrad(prec, df, w1, np_, cc, n, size, size)
    assert torch.isfinite(dx).all(), "an input pixel of x was never written"
    got = [dx]
    want = [ref[:, :1]]
    if cc:
        assert torch.isfinite(dpl).all(), "an input pixel of the planes was never written"
        got.append(dpl)
        want.append(ref[:, 1:].sum(0, keepdim=True) if shared else ref[:, 1:])
    again = run_stem_dgrad(prec, df, w1, np_, cc, n, size, size)
    assert torch.equal(dx, again[0]) and (dpl is None or torch.equal(dpl, again[1])), "the stem data gradient is not deterministic"
    err = rel_l2(torch.cat([g.flatten() for g in got]).double(), torch.cat([g.flatten() for g in want]))
    print(f"stem dgrad [{prec}] cin={cin} np={np_} {size}x{size}: rel-L2 {err:.2e} (gate {KERNEL_GATE[prec]:.0e})")
    assert err < KERNEL_GATE[prec]


def test_stem_dgrad_tc_kernel_is_tensor_core_code():
    import __graft_entry__ as ge
    from sbgm_danra_b200 import _lib
    cuobjdump = shutil.which("cuobjdump") or shutil.which("cuobjdump", path=os.path.dirname(ge.NVCC))
    if cuobjdump is None or not os.path.exists(_lib.LIB_PATH):
        pytest.skip("cuobjdump or library unavailable")
    sass = subprocess.run([cuobjdump, "-sass", _lib.LIB_PATH], capture_output=True, text=True).stdout
    blocks = [b for b in sass.split("Function : ") if b.startswith("_ZN4sbgm20stem_dgrad_tc_kernel")]
    assert len(blocks) == 2, "expected the bf16 and split-bf16 instances of stem_dgrad_tc_kernel"
    for b in blocks:
        assert "UTCHMMA" in b and "LDTM" in b


# ---- 2.-6. the network -------------------------------------------------------------------------------------------------
CONFIGS = {"cin2": dict(n_lr=1), "cin7_seasons": dict(n_lr=2, geo=True, seasons=True)}


def _case(config, batch=4, size=64, shared=False):
    from oracle.synth import config_for, synth_batch, synth_state_dict
    ck = CONFIGS[config]
    cfg = config_for(**ck)
    b = synth_batch(batch=batch, size=size, shared_cond=shared, **ck)
    t = torch.linspace(0.2, 0.9, batch)
    v = gen(batch, 1, size, size, seed=77)
    return cfg, synth_state_dict(cfg), b, t, v


def _inputs(b):
    return [("x", b.x), ("cond_img", b.cond_img), ("lsm_cond", b.lsm_cond), ("topo_cond", b.topo_cond)]


def _leaf_inputs(b, shared):
    return {k: (a[:1] if shared and k == "cond_img" else a).clone() for k, a in _inputs(b) if a is not None}


@functools.lru_cache(maxsize=None)
def _oracle_vjp(config, bn_train, autocast=False, batch=4, size=64, shared=False, dtype=torch.float32):
    from oracle import score_ref
    cfg, sd, b, t, v = _case(config, batch, size, shared)
    sd = {k: (a.to(dtype) if a.is_floating_point() else a) for k, a in sd.items()}
    leaves = {k: a.to(dtype).requires_grad_() for k, a in _leaf_inputs(b, shared).items()}
    args = {k: leaves.get(k) for k, _ in _inputs(b)}
    if shared:
        args["cond_img"] = leaves["cond_img"].expand(batch, *leaves["cond_img"].shape[1:])
    with torch.autocast("cpu", dtype=torch.bfloat16, enabled=autocast):
        score = score_ref.score_forward(sd, cfg, args["x"], t.to(dtype), b.y, args["cond_img"], args["lsm_cond"], args["topo_cond"],
                                        bn_train=bn_train)
    names = sorted(leaves)
    grads = torch.autograd.grad(score.to(dtype), [leaves[k] for k in names], v.to(dtype))
    return {k: g.double() for k, g in zip(names, grads)}


def _ours_vjp(config, precision, bn_train, pre, frozen=False, batch=4, size=64, shared=False):
    from sbgm_danra_b200._smoke import build_model
    cfg, sd, b, t, v = _case(config, batch, size, shared)
    net = build_model(cfg, sd, precision, DEV)
    net.train(bn_train)
    net.debug_pre_sigma_div = pre
    if frozen:
        net.requires_grad_(False)
    leaves = {k: a.to(DEV).requires_grad_() for k, a in _leaf_inputs(b, shared).items()}
    score = net(leaves["x"], t.to(DEV), None if b.y is None else b.y.to(DEV), leaves.get("cond_img"), leaves.get("lsm_cond"),
                leaves.get("topo_cond"))
    names = sorted(leaves)
    grads = torch.autograd.grad(score, [leaves[k] for k in names], v.to(DEV))
    return net, {k: g.cpu().double() for k, g in zip(names, grads)}


def _whole(got, want):
    keys = sorted(want)
    assert sorted(got) == keys
    return rel_l2(torch.cat([got[k].flatten() for k in keys]), torch.cat([want[k].flatten() for k in keys]))


def _gate(config, precision, bn_train, **kw):
    want = _oracle_vjp(config, bn_train, dtype=torch.float64, **kw)
    fp32 = 2 * _whole(_oracle_vjp(config, bn_train, **kw), want)
    if precision == "fp32":
        return want, max(NET_GATE[precision], fp32)
    autocast = _whole(_oracle_vjp(config, bn_train, autocast=True, **kw), want)
    if precision == "bf16":
        return want, 2 * autocast
    return want, max(NET_GATE[precision], fp32, SPLIT_FRACTION_OF_AUTOCAST * autocast)


def _check(config, precision, bn_train, got, **kw):
    want, gate = _gate(config, precision, bn_train, **kw)
    err = _whole(got, want)
    print(f"input VJP {config} [{precision}] bn_train={bn_train} {kw}: rel-L2 {err:.2e} (gate {gate:.1e})")
    assert err < gate


@pytest.mark.parametrize("precision", ["fp32", "bf16x3", "fp16x2", "bf16"])
@pytest.mark.parametrize("pre", [True, False])
@pytest.mark.parametrize("bn_train", [False, True])
@pytest.mark.parametrize("config", list(CONFIGS))
def test_input_vjp_matches_oracle(config, bn_train, pre, precision):
    _, got = _ours_vjp(config, precision, bn_train, pre)
    _check(config, precision, bn_train, got)


def test_input_vjp_at_c4_launch_shape():
    """bench.py's C4 shape: batch 64, 128x128, Cin = 7 + seasons; frozen model, running-statistics BatchNorm."""
    kw = dict(batch=64, size=128)
    _, got = _ours_vjp("cin7_seasons", "bf16x3", False, False, frozen=True, **kw)
    _check("cin7_seasons", "bf16x3", False, got, **kw)


@pytest.mark.parametrize("precision", ["fp32", "bf16x3"])
def test_shared_conditioning_gradient_is_the_batch_sum(precision):
    _, got = _ours_vjp("cin2", precision, False, False, shared=True)
    assert got["cond_img"].shape[0] == 1
    _check("cin2", precision, False, got, shared=True)


@pytest.mark.parametrize("precision", ["fp32", "bf16x3"])
def test_frozen_model_runs_data_gradients_only(monkeypatch, precision):
    from sbgm_danra_b200 import engine, train_engine
    monkeypatch.setenv("SBGM_B200_TRAIN_GRAPHS", "0")
    seen, recording = [], [False]
    for mod in (engine, train_engine):
        orig = mod.call

        def wrapped(name, *args, _orig=orig):
            if recording[0]:
                seen.append(name)
            return _orig(name, *args)
        monkeypatch.setattr(mod, "call", wrapped)
    from sbgm_danra_b200._smoke import build_model
    cfg, sd, b, t, v = _case("cin7_seasons")
    net = build_model(cfg, sd, precision, DEV).requires_grad_(False)
    x = b.x.clone().to(DEV).requires_grad_()
    score = net(x, t.to(DEV), b.y.to(DEV), b.cond_img.to(DEV), b.lsm_cond.to(DEV), b.topo_cond.to(DEV))
    recording[0] = True
    (dx,) = torch.autograd.grad(score, [x], v.to(DEV))
    recording[0] = False
    assert all(p.grad is None for p in net.parameters())
    assert seen and not (set(seen) & PARAM_ONLY), f"parameter-only launches in a frozen backward: {sorted(set(seen) & PARAM_ONLY)}"
    assert ("sbgm_stem_dgrad_simt" if precision == "fp32" else "sbgm_stem_dgrad_tc") in seen
    want, gate = _gate("cin7_seasons", precision, False)
    err = rel_l2(dx.cpu().double(), want["x"])
    print(f"frozen [{precision}]: dx rel-L2 {err:.2e} (gate {gate:.1e}), {len(seen)} launches in backward")
    assert err < gate


@pytest.mark.parametrize("precision", ["fp32", "bf16x3"])
def test_mixed_request_keeps_parameter_gradients_bit_identical(precision):
    from sbgm_danra_b200._smoke import build_model
    cfg, sd, b, t, v = _case("cin7_seasons")
    net = build_model(cfg, sd, precision, DEV).train()
    cond = [a.to(DEV) for a in (b.y, b.cond_img, b.lsm_cond, b.topo_cond)]

    def step(x_grad):
        net.zero_grad(set_to_none=True)
        x = b.x.clone().to(DEV).requires_grad_(x_grad)
        (net(x, t.to(DEV), *cond) * v.to(DEV)).sum().backward()
        return x.grad, {k: p.grad.clone() for k, p in net.named_parameters() if p.grad is not None}

    sd_state = {k: s.clone() for k, s in net.state_dict().items()}
    xg0, plain = step(False)
    net.load_state_dict(sd_state)                 # the same running statistics for both steps
    xg1, mixed = step(True)
    assert xg0 is None and xg1 is not None and torch.isfinite(xg1).all()
    assert sorted(plain) == sorted(mixed)
    for k in plain:
        assert torch.equal(plain[k], mixed[k]), k


def test_graph_replay_matches_eager(monkeypatch):
    from sbgm_danra_b200._smoke import build_model
    cfg, sd, b, t, v = _case("cin7_seasons")
    net = build_model(cfg, sd, "bf16x3", DEV).requires_grad_(False)
    cond = [a.to(DEV) for a in (b.y, b.cond_img, b.lsm_cond, b.topo_cond)]
    xs = [(b.x * (1 + 0.1 * k)).to(DEV) for k in range(4)]

    def vjp(x):
        x = x.clone().requires_grad_()
        lsm = cond[2].clone().requires_grad_()
        gx, gl = torch.autograd.grad(net(x, t.to(DEV), cond[0], cond[1], lsm, cond[3]), [x, lsm], v.to(DEV))
        return gx, gl

    graphed = [vjp(x) for x in xs]
    runner = next(iter(net._train_runners.values()))
    assert runner.g_bwd is not None, "calls 3 and 4 were not replayed from the captured graphs"
    third = [g.clone() for g in graphed[2]]
    graphed_again = vjp(xs[3])              # a fifth call: the third call's gradients must survive it too
    assert all(torch.equal(a, c) for a, c in zip(graphed[2], third)), "a later replay overwrote an earlier call's gradient"
    monkeypatch.setenv("SBGM_B200_TRAIN_GRAPHS", "0")
    net._train_runners.clear()
    for k in (2, 3):
        eager = vjp(xs[k])
        assert all(torch.equal(a, c) for a, c in zip(graphed[k], eager)), f"call {k + 1}: replay differs from the eager engine"
    assert all(torch.equal(a, c) for a, c in zip(graphed_again, graphed[3]))
