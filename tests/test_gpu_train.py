"""GPU parity tests of the DSM training path: every backward kernel against torch autograd on the same
operator (plain fp32 torch), then the whole loss + gradients against the CPU oracle's autograd and the
committed reference goldens (tests/golden/, generated from the real reference by make_golden.py).

Tolerances are relative L2: fp32 kernels 2e-5; bf16x3 (split-bf16 tensor cores, fp32-class) 2e-4 per op and
2e-3 for whole-network gradients; bf16 5e-2 per op (reported, bf16 gradients are bf16-rounded)."""
import json
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import GOLDEN_DIR, rel_l2

pytestmark = pytest.mark.gpu

FMTS = {"fp32": 0, "bf16": 1, "bf16x3": 2}
TOL = {"fp32": 2e-5, "bf16": 5e-2, "bf16x3": 2e-4}
DEV = "cuda:0"
ACT = {"none": 0, "relu": 1, "silu": 2, "gelu": 3}
ACT_F = {"none": lambda v: v, "relu": F.relu, "silu": F.silu, "gelu": F.gelu}


def gen(*shape, seed=0, scale=1.0):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed)) * scale


@pytest.fixture(scope="module")
def E():
    from sbgm_danra_b200 import engine
    return engine


@pytest.fixture(scope="module")
def T():
    from sbgm_danra_b200 import train_engine
    return train_engine


def act_of(E, x, fmt):
    return E.Act.from_nchw(x.to(DEV), fmt)


def stored(E, x, fmt):
    """x after a round trip through the activation storage format (what the kernels actually see)."""
    return act_of(E, x, fmt).to_nchw().cpu()


def make_tk(T, fmt):
    grads = {}

    def flat(name, shape):
        grads[name] = torch.zeros(shape, dtype=torch.float32, device=DEV)
        return grads[name]

    tk = T.TrainKernels(fmt, torch.device(DEV), flat)
    tk.tape = T.Tape(fmt, torch.device(DEV))
    return tk, grads


def run_tape(tk):
    for fn in reversed(tk.tape.steps):
        fn()


# ---- normalisation ---------------------------------------------------------------------------------
@pytest.mark.parametrize("prec", ["fp32", "bf16x3"])
@pytest.mark.parametrize("shape", [(3, 64, 8), (5, 128, 48)])        # the second one splits every sample over several chunk blocks
@pytest.mark.parametrize("case", ["bn_train_relu_res_tproj", "bn_eval", "gn_silu_skip_tproj", "gn_plain", "instance_relu"])
def test_norm_forward_backward(E, T, prec, case, shape):
    fmt = FMTS[prec]
    n, c, h = shape
    x0, add0, dy0 = gen(n, c, h, h, seed=1), gen(n, c, h, h, seed=2), gen(n, c, h, h, seed=3)
    gamma, beta = 1 + 0.2 * gen(c, seed=4), 0.1 * gen(c, seed=5)
    tproj = gen(n, 2 * c, seed=6)[:, c:]           # a column slice (stride 2c), like the real projection table
    x, add, dy = (stored(E, v, fmt).requires_grad_(v is not dy0) for v in (x0, add0, dy0))
    g, b = gamma.clone().requires_grad_(), beta.clone().requires_grad_()
    tp = tproj.clone().requires_grad_()
    tk, grads = make_tk(T, fmt)
    xa, adda = act_of(E, x.detach(), fmt), act_of(E, add.detach(), fmt)
    tpc = tproj.to(DEV)
    tpj = torch.zeros(n, 2 * c, device=DEV)
    tpj[:, c:] = tpc
    tp_dev = tpj[:, c:]
    dtp = torch.zeros(n, 2 * c, device=DEV)
    rm, rv = gen(c, seed=7) * 0.1, torch.rand(c, generator=torch.Generator().manual_seed(8)) + 0.5
    if case == "bn_train_relu_res_tproj":
        bn = dict(weight=gamma.to(DEV), bias=beta.to(DEV), running_mean=rm.to(DEV), running_var=rv.to(DEV), weight_name="g", bias_name="b")
        ya = tk.batchnorm(xa, bn, True, act=ACT["relu"], residual=adda, tproj=tp_dev, dtproj=dtp[:, c:])
        rm_ref, rv_ref = rm.clone(), rv.clone()
        want = F.relu(F.batch_norm(x, rm_ref, rv_ref, g, b, training=True, momentum=0.1, eps=1e-5) + add) + tp[:, :, None, None]
        assert rel_l2(bn["running_mean"].cpu(), rm_ref) < 1e-5 and rel_l2(bn["running_var"].cpu(), rv_ref) < 1e-5
    elif case == "bn_eval":
        bn = dict(weight=gamma.to(DEV), bias=beta.to(DEV), running_mean=rm.to(DEV), running_var=rv.to(DEV), weight_name="g", bias_name="b")
        ya = tk.batchnorm(xa, bn, False, act=ACT["relu"])
        want = F.relu(F.batch_norm(x, rm, rv, g, b, training=False, eps=1e-5))
    elif case == "gn_silu_skip_tproj":
        ya = tk.groupnorm(xa, gamma.to(DEV), beta.to(DEV), "g", "b", 8, act=ACT["silu"], skip=adda, tproj=tp_dev, dtproj=dtp[:, c:],
                          prev_bias="pb")
        want = F.silu(F.group_norm(x, 8, g, b, eps=1e-5) + add + tp[:, :, None, None])
    elif case == "gn_plain":
        ya = tk.groupnorm(xa, gamma.to(DEV), beta.to(DEV), "g", "b", 8, prev_bias="pb")
        want = F.group_norm(x, 8, g, b, eps=1e-5)
    else:
        ya = tk.groupnorm(xa, None, None, None, None, c, act=ACT["relu"], skip=adda)
        want = F.relu(F.instance_norm(x, eps=1e-5) + add)
    assert rel_l2(ya.to_nchw().cpu(), want.detach()) < max(TOL[prec], 1e-4 if prec != "fp32" else 0)
    want.backward(dy)
    tk.tape.add(ya, act_of(E, dy, fmt))
    run_tape(tk)
    tol = TOL[prec] * 5
    assert rel_l2(tk.tape.grads[xa.buf.data_ptr()].to_nchw().cpu(), x.grad) < tol
    if add.grad is not None:
        assert rel_l2(tk.tape.grads[adda.buf.data_ptr()].to_nchw().cpu(), add.grad) < tol
    if g.grad is not None:
        assert rel_l2(grads["g"].cpu(), g.grad) < tol and rel_l2(grads["b"].cpu(), b.grad) < tol
    if tp.grad is not None:
        assert rel_l2(dtp[:, c:].cpu(), tp.grad) < tol
    if "pb" in grads:       # bias gradient of the convolution in front of the norm = dx summed over n, h, w (closed form in the kernel)
        assert rel_l2(grads["pb"].cpu(), x.grad.sum(dim=(0, 2, 3))) < tol * 4
    # the reduction's tickets are left zero, so the same scratch serves the next layer
    from sbgm_danra_b200 import _lib
    assert int(tk._scratch["norm_bwd"][:4096].view(torch.int32).abs().sum()) == 0


@pytest.mark.parametrize("prec", ["fp32", "bf16x3"])
def test_layernorm_act_upsample_backward(E, T, prec):
    fmt = FMTS[prec]
    tk, grads = make_tk(T, fmt)
    # LayerNorm over tokens [1, 1, rows, c]
    rows, c = 200, 256
    x = stored(E, gen(1, c, 1, rows, seed=1), fmt).requires_grad_()
    dy = stored(E, gen(1, c, 1, rows, seed=2), fmt)
    gamma, beta = (1 + 0.2 * gen(c, seed=3)).requires_grad_(), (0.1 * gen(c, seed=4)).requires_grad_()
    xa = act_of(E, x.detach(), fmt)
    ya = tk.layernorm(xa, gamma.detach().to(DEV), beta.detach().to(DEV), "g", "b")
    want = F.layer_norm(x.permute(0, 2, 3, 1), (c,), gamma, beta, eps=1e-5).permute(0, 3, 1, 2)
    want.backward(dy)
    tk.tape.add(ya, act_of(E, dy, fmt))
    run_tape(tk)
    assert rel_l2(tk.tape.grads[xa.buf.data_ptr()].to_nchw().cpu(), x.grad) < TOL[prec] * 5
    assert rel_l2(grads["g"].cpu(), gamma.grad) < TOL[prec] * 5 and rel_l2(grads["b"].cpu(), beta.grad) < TOL[prec] * 5
    # activations
    for name in ("relu", "silu", "gelu"):
        tk, _ = make_tk(T, fmt)
        x = stored(E, gen(2, 64, 5, 7, seed=5), fmt).requires_grad_()
        dy = stored(E, gen(2, 64, 5, 7, seed=6), fmt)
        xa = act_of(E, x.detach(), fmt)
        ya = tk.activation(xa, ACT[name])
        want = ACT_F[name](x)
        assert rel_l2(ya.to_nchw().cpu(), want.detach()) < max(TOL[prec], 1e-5)
        want.backward(dy)
        tk.tape.add(ya, act_of(E, dy, fmt))
        run_tape(tk)
        assert rel_l2(tk.tape.grads[xa.buf.data_ptr()].to_nchw().cpu(), x.grad) < TOL[prec] * 2, name
    # bilinear x2 upsample
    for shape in ((2, 64, 4, 4), (1, 72, 5, 9)):
        tk, _ = make_tk(T, fmt)
        x = stored(E, gen(*shape, seed=7), fmt).requires_grad_()
        dy = stored(E, gen(shape[0], shape[1], 2 * shape[2], 2 * shape[3], seed=8), fmt)
        xa = act_of(E, x.detach(), fmt)
        ya = tk.upsample2x(xa)
        want = F.interpolate(x, scale_factor=2, mode="bilinear", align_corners=False)
        want.backward(dy)
        tk.tape.add(ya, act_of(E, dy, fmt))
        run_tape(tk)
        assert rel_l2(tk.tape.grads[xa.buf.data_ptr()].to_nchw().cpu(), x.grad) < TOL[prec] * 2, shape


@pytest.mark.parametrize("prec", ["fp32", "bf16x3", "bf16"])
@pytest.mark.parametrize("b,s,c,heads", [(2, 16, 128, 4), (3, 64, 256, 4), (1, 100, 64, 8),
                                         # bf16: the one-launch tensor-core kernel (attention_bwd_mma.cu) -- head dim 128 / 16-token
                                         # chunks, head dim 32 / 64-token chunks over two warps' worth of slabs, S = 48 (16-token chunks)
                                         (2, 16, 512, 4), (2, 256, 128, 4), (1, 48, 128, 4)])
def test_attention_backward(E, T, prec, b, s, c, heads):
    fmt = FMTS[prec]
    tk, _ = make_tk(T, fmt)
    qkv = stored(E, gen(1, 3 * c, 1, b * s, seed=1), fmt).requires_grad_()
    dy = stored(E, gen(1, c, 1, b * s, seed=2), fmt)
    qa = act_of(E, qkv.detach(), fmt)
    ya = tk.attention_core(qa, b, s, c, heads)
    tok = qkv[0, :, 0, :].t().reshape(b, s, 3 * c)
    q, k, v = (z.reshape(b, s, heads, c // heads).permute(0, 2, 1, 3) for z in tok.chunk(3, dim=-1))
    att = torch.softmax(q @ k.transpose(-1, -2) / (c // heads) ** 0.5, dim=-1) @ v
    want = att.permute(0, 2, 1, 3).reshape(b * s, c).t()[None, :, None, :]
    assert rel_l2(ya.to_nchw().cpu(), want.detach()) < max(TOL[prec], 2e-5)
    want.backward(dy)
    tk.tape.add(ya, act_of(E, dy, fmt))
    run_tape(tk)
    got = tk.tape.grads[qa.buf.data_ptr()].to_nchw().cpu()
    if prec == "bf16":      # per q / k / v block: P and dS are rounded to bfloat16 between the products (as in flash attention)
        for i, name in enumerate("qkv"):
            e = rel_l2(got[:, i * c:(i + 1) * c], qkv.grad[:, i * c:(i + 1) * c])
            assert e < 2e-2, (name, e)
    else:
        assert rel_l2(got, qkv.grad) < TOL[prec] * 5


# ---- convolution gradients ----------------------------------------------------------------------------
CONV_CASES = [
    # n, h, w, cin, cout, k, stride, pad, bias
    (2, 16, 16, 64, 64, 3, 1, 1, True),        # c64 kernel path (dgrad) + wgrad
    (2, 8, 8, 128, 256, 3, 1, 1, True),
    (2, 16, 16, 64, 128, 3, 2, 1, False),      # strided 3x3: parity-sliced dgrad
    (2, 16, 16, 128, 256, 1, 2, 0, False),     # downsample 1x1 stride 2
    (2, 32, 32, 64, 64, 8, 2, 3, False),       # Encoder.conv2
    (3, 4, 4, 512, 512, 3, 1, 1, True),        # tiny maps, tile covers several images
    (1, 1, 300, 256, 768, 1, 1, 0, True),      # Linear (token matrix, ragged tail)
]


@pytest.mark.parametrize("prec", ["fp32", "bf16x3", "bf16"])
@pytest.mark.parametrize("case", CONV_CASES)
def test_conv_backward(E, T, prec, case):
    fmt = FMTS[prec]
    n, h, w, cin, cout, k, stride, pad, bias = case
    wt = gen(cout, cin, k, k, seed=1, scale=(cin * k * k) ** -0.5)
    bt = gen(cout, seed=2, scale=0.1) if bias else None
    x = stored(E, gen(n, cin, h, w, seed=3), fmt).requires_grad_()
    ho, wo = (h + 2 * pad - k) // stride + 1, (w + 2 * pad - k) // stride + 1
    dy = stored(E, gen(n, cout, ho, wo, seed=4), fmt)
    wr = wt.clone().requires_grad_()
    br = bt.clone().requires_grad_() if bias else None
    want = F.conv2d(x, wr, br, stride=stride, padding=pad)
    want.backward(dy)
    tk, grads = make_tk(T, fmt)
    layer = T.ConvLayer("w", wt.to(DEV), None if bt is None else bt.to(DEV), fmt, "b" if bias else None)
    xa = act_of(E, x.detach(), fmt)
    ya = tk.conv(xa, layer, stride=stride, pad=pad)
    ftol = {"fp32": 2e-5, "bf16x3": 1e-4, "bf16": 2e-2}[prec]
    assert rel_l2(ya.to_nchw().cpu(), want.detach()) < ftol
    tk.tape.add(ya, act_of(E, dy, fmt))
    run_tape(tk)
    e_dx = rel_l2(tk.tape.grads[xa.buf.data_ptr()].to_nchw().cpu(), x.grad)
    # dW is fp32 sums of exact products of the stored x and dy (bf16x3 drops lo x lo, ~2^-16): gated against float64, not
    # at ftol.  dx is rounded to the activation format on output, so it keeps the forward's gate.
    dw_ref = torch.nn.grad.conv2d_weight(x.detach().double(), wt.shape, dy.double(), stride=stride, padding=pad)
    e_dw = rel_l2(grads["w"].cpu(), dw_ref)
    print(f"{case} [{prec}] dx {e_dx:.2e} dW {e_dw:.2e}")
    assert e_dx < ftol and e_dw < {"fp32": 1e-5, "bf16x3": 5e-5, "bf16": 1e-5}[prec]
    if bias:
        assert rel_l2(grads["b"].cpu(), br.grad) < ftol


@pytest.mark.parametrize("prec", ["fp32", "bf16x3"])
@pytest.mark.parametrize("cc,bcast", [(1, False), (6, True)])
def test_stem_wgrad(E, prec, cc, bcast):
    from sbgm_danra_b200 import _lib
    from sbgm_danra_b200._lib import call
    fmt = FMTS[prec]
    n, h = 3, 32
    x = gen(n, 1, h, h, seed=1)
    planes = gen(1 if bcast else n, cc, h, h, seed=2)
    w = gen(64, cc + 1, 8, 8, seed=3, scale=0.1).requires_grad_()
    full = torch.cat([x, planes.expand(n, -1, -1, -1)], 1)
    df = stored(E, gen(n, 64, h // 2, h // 2, seed=4), fmt)
    F.conv2d(full, w, None, stride=2, padding=3).backward(df)
    dfa = act_of(E, df, fmt)
    dw = torch.zeros(64, cc + 1, 8, 8, device=DEV)
    ws = torch.empty(_lib.query("sbgm_stem_wgrad_workspace_floats", cc + 1), device=DEV)
    xd, pd = x.to(DEV).contiguous(), planes.to(DEV).contiguous()
    call("sbgm_stem_wgrad", xd.data_ptr(), pd.data_ptr(), pd.shape[0], cc, dfa.ptr, dfa.plane, fmt, dw.data_ptr(), n, h, h,
         ws.data_ptr(), torch.cuda.current_stream().cuda_stream)
    assert rel_l2(dw.cpu(), w.grad) < 2e-5


@pytest.mark.parametrize("prec", ["fp32", "bf16x3", "bf16"])
@pytest.mark.parametrize("geom", [(3, 16, 24, 64), (2, 13, 37, 64), (2, 9, 9, 256), (2, 16, 16, 24)])
def test_final_conv_backward(E, prec, geom):
    """(n, h, w, c): ragged tiles, one pixel lane per warp (c = 256), and c / 8 not a power of two (the two-kernel fall-back)."""
    from sbgm_danra_b200 import _lib
    from sbgm_danra_b200._lib import call
    fmt = FMTS[prec]
    n, h, w, c = geom
    fused = c in (64, 128, 256)
    a = stored(E, gen(n, c, h, w, seed=1), fmt).requires_grad_()
    wt = gen(1, c, 3, 3, seed=2, scale=0.05).requires_grad_()
    bt = gen(1, seed=3).requires_grad_()
    inv = torch.rand(n, generator=torch.Generator().manual_seed(4)) + 0.5
    ds = gen(n, 1, h, w, seed=5)
    (F.conv2d(a, wt, bt, padding=1) * inv[:, None, None, None]).backward(ds)
    aa = act_of(E, a.detach(), fmt)
    da = E.Act(fmt, n, h, w, c, torch.device(DEV))
    dw, db = torch.zeros(1, c, 3, 3, device=DEV), torch.zeros(1, device=DEV)
    wp = wt.detach().permute(0, 2, 3, 1).reshape(9, c).contiguous().to(DEV)
    ws = torch.empty(_lib.query("sbgm_final_conv_backward_scratch_floats", c), device=DEV)
    dsd, invd = ds.to(DEV), inv.to(DEV)
    dbu = torch.zeros(c, device=DEV) if fused else None
    call("sbgm_final_conv_backward", dsd.data_ptr(), invd.data_ptr(), aa.ptr, aa.plane, fmt, wp.data_ptr(), da.ptr, da.plane,
         dw.data_ptr(), db.data_ptr(), None if dbu is None else dbu.data_ptr(), n, h, w, c, ws.data_ptr(),
         torch.cuda.current_stream().cuda_stream)
    assert rel_l2(da.to_nchw().cpu(), a.grad) < TOL[prec]
    assert rel_l2(dw.cpu(), wt.grad) < 2e-5 and rel_l2(db.cpu(), bt.grad) < 2e-5
    if fused:           # bias gradient of the convolution that produced `a`: da summed over n, h, w
        assert rel_l2(dbu.cpu(), a.grad.sum(dim=(0, 2, 3))) < 2e-5


def test_time_embed_backward(E):
    from oracle import score_ref
    from sbgm_danra_b200 import _lib
    from sbgm_danra_b200._lib import call
    te, rows = 256, 5
    tp = E.TimeProjector(torch.device(DEV), te)
    W0, W1 = gen(128, seed=1, scale=30.0), gen(128, seed=2, scale=30.0)
    s0, s1 = tp.add_set(W0.to(DEV)), tp.add_set(W1.to(DEV))
    heads = [("a", s0, 64), ("b", s1, 128), ("c", s0, 256)]
    ws = {}
    for i, (name, s, c) in enumerate(heads):
        ws[name] = (gen(c, te, seed=10 + i, scale=0.06).requires_grad_(), gen(c, seed=20 + i, scale=0.1).requires_grad_())
        tp.add_head(name, s, ws[name][0].detach().to(DEV), ws[name][1].detach().to(DEV))
    lab = gen(5, te, seed=30, scale=0.5).requires_grad_()
    tp.label_emb = lab.detach().to(DEV)
    tp.finalize()
    t = torch.rand(rows, generator=torch.Generator().manual_seed(3))
    y = torch.tensor([1, 4, 0, 1, 2])
    dout = gen(rows, tp.c_total, seed=40)
    outs = []
    for name, s, c in heads:
        emb = score_ref.fourier_embed(W0 if s == s0 else W1, t)
        if s == s0:
            emb = emb + lab[y]
        outs.append(F.linear(F.silu(emb), *ws[name]))
    torch.cat(outs, 1).backward(dout)
    fw, pw, pb, ps = tp._packed
    dpw, dpb, dlab = torch.empty_like(pw), torch.empty_like(pb), torch.zeros(5, te, device=DEV)
    scratch = torch.empty(_lib.query("sbgm_time_embed_backward_scratch_floats", 2, te, rows), device=DEV)
    td, yd, dd = t.to(DEV), y.to(DEV), dout.to(DEV)
    call("sbgm_time_embed_backward", dd.data_ptr(), td.data_ptr(), yd.data_ptr(), fw.data_ptr(), 2, te, tp.label_emb.data_ptr(), 5,
         pw.data_ptr(), ps.data_ptr(), tp.c_total, rows, dpw.data_ptr(), dpb.data_ptr(), dlab.data_ptr(), scratch.data_ptr(),
         torch.cuda.current_stream().cuda_stream)
    assert rel_l2(dpw.cpu(), torch.cat([ws[n][0].grad for n, _, _ in heads])) < 2e-5
    assert rel_l2(dpb.cpu(), torch.cat([ws[n][1].grad for n, _, _ in heads])) < 2e-5
    assert rel_l2(dlab.cpu(), lab.grad) < 2e-5


# ---- whole network: loss + gradients ----------------------------------------------------------------------
def _dsm_case(precision, mode, size=32, batch=4):
    from oracle import philox_ref, score_ref
    from oracle.synth import config_for, synth_batch, synth_state_dict
    from sbgm_danra_b200 import score_sampling
    from sbgm_danra_b200._smoke import build_model
    from sbgm_danra_b200.score_unet import loss_fn, marginal_prob_std_fn
    cfg = config_for(n_lr=2, geo=True, seasons=True)
    sd = synth_state_dict(cfg)
    b = synth_batch(batch=batch, size=size, n_lr=2, geo=True, seasons=True)
    net = build_model(cfg, sd, precision, DEV)
    net.train(mode == "train")
    score_sampling.manual_seed(2024)
    c = lambda v: None if v is None else v.to(DEV)
    loss = loss_fn(net, c(b.x), marginal_prob_std_fn, y=c(b.y), cond_img=c(b.cond_img), lsm_cond=c(b.lsm_cond),
                   topo_cond=c(b.topo_cond), sdf_cond=c(b.sdf_cond))
    loss.backward()
    # oracle with the same Philox draws
    sdo = {k: (v.clone().requires_grad_() if v.is_floating_point() and not k.endswith(("running_mean", "running_var", ".W")) else v.clone())
           for k, v in sd.items()}
    u = torch.from_numpy(philox_ref.uniform(batch, 2024, philox_ref.DRAW_DSM_T))
    z = torch.from_numpy(philox_ref.normal(b.x.numel(), 2024, philox_ref.DRAW_DSM_Z)).reshape(b.x.shape)
    rt = u * (1.0 - 1e-3) + 1e-3
    lo = score_ref.dsm_loss(sdo, cfg, b.x, rt, z, b.y, b.cond_img, b.lsm_cond, b.topo_cond, b.sdf_cond, bn_train=(mode == "train"))
    lo.backward()
    return net, loss, sdo, lo


@pytest.mark.parametrize("precision", ["fp32", "bf16x3", "bf16"])
@pytest.mark.parametrize("mode", ["train", "eval"])
def test_dsm_loss_and_gradients_match_oracle(golden, precision, mode):
    net, loss, sdo, lo = _dsm_case(precision, mode)
    ltol = {"fp32": 1e-4, "bf16x3": 1e-3, "bf16": 5e-2}[precision]
    # bf16 stores every activation AND every activation gradient in bf16; at this test's size (batch 4, 32x32: the deep
    # BatchNorm layers normalise over 4..16 values) single small tensors can be off by tens of percent, so bf16 is gated on
    # the whole gradient vector (below) and reported per tensor
    gtol = {"fp32": 1e-3, "bf16x3": 2e-3, "bf16": 6e-1}[precision]
    assert abs(loss.item() - lo.item()) / abs(lo.item()) < ltol
    assert abs(loss.item() - float(golden[f"dsm_{mode}/loss"])) / abs(float(golden[f"dsm_{mode}/loss"])) < ltol
    worst = ("", 0.0)
    params = dict(net.named_parameters())
    unused = []
    for k, v in sdo.items():
        if not (torch.is_tensor(v) and v.requires_grad):
            continue
        if v.grad is None:
            unused.append(k)
            assert params[k].grad is None, f"{k} unused by the oracle but has a gradient here"
            continue
        assert params[k].grad is not None, f"{k} has no gradient"
        e = rel_l2(params[k].grad.cpu(), v.grad)
        if e > worst[1]:
            worst = (k, e)
        assert precision == "bf16" or e < gtol, f"{k}: rel-L2 {e:.3e}"
    used = [k for k, v in sdo.items() if torch.is_tensor(v) and v.requires_grad and v.grad is not None]
    whole = rel_l2(torch.cat([params[k].grad.cpu().reshape(-1) for k in used]), torch.cat([sdo[k].grad.reshape(-1) for k in used]))
    print(f"[{precision}/{mode}] loss {loss.item():.6f} vs oracle {lo.item():.6f}; whole-gradient rel-L2 {whole:.2e}; "
          f"worst tensor {worst[0]} {worst[1]:.2e}; unused {len(unused)}")
    assert whole < {"fp32": 1e-4, "bf16x3": 1e-3, "bf16": 2.5e-1}[precision]   # bf16 at batch 4 / 32x32: 1.4e-1 (train), reported
    if precision == "bf16":
        return
    with open(os.path.join(GOLDEN_DIR, "dsm_grad_keys.json")) as f:
        gkeys = json.load(f)
    got = np.array([params[k].grad.norm().item() for k in gkeys])
    assert np.allclose(got, golden[f"dsm_{mode}/grad_norms"], rtol=gtol)
    assert rel_l2(params["decoder.final_layer.conv.weight"].grad.cpu(), golden[f"dsm_{mode}/grad_final_conv"]) < gtol


def test_bn_running_stats_and_training_steps_reduce_loss():
    """Three Adam steps on a fixed batch: the running statistics move as torch's would and the loss falls."""
    from oracle.synth import config_for, synth_batch, synth_state_dict
    from sbgm_danra_b200 import score_sampling
    from sbgm_danra_b200._smoke import build_model
    from sbgm_danra_b200.score_unet import loss_fn, marginal_prob_std_fn
    cfg = config_for(n_lr=1)
    net = build_model(cfg, synth_state_dict(cfg), "bf16x3", DEV).train()
    b = synth_batch(batch=4, size=32, n_lr=1)
    opt = torch.optim.Adam(net.parameters(), lr=1e-4)
    nbt0 = int(net.encoder.bn1.num_batches_tracked)
    rm0 = net.encoder.bn1.running_mean.clone()
    losses = []
    for _ in range(4):
        score_sampling.manual_seed(11)                 # same (t, z): a deterministic objective
        opt.zero_grad()
        loss = loss_fn(net, b.x.to(DEV), marginal_prob_std_fn, cond_img=b.cond_img.to(DEV), sdf_cond=b.sdf_cond.to(DEV))
        loss.backward()
        opt.step()
        losses.append(loss.item())
    assert int(net.encoder.bn1.num_batches_tracked) == nbt0 + 4
    assert not torch.equal(net.encoder.bn1.running_mean, rm0)
    assert losses[-1] < losses[0], losses
    assert all(np.isfinite(losses))


def test_graph_replay_reproduces_eager_step_bitwise():
    """Steps 1-2 run the eager engine, steps 3+ replay the captured forward / backward CUDA graphs
    (train_engine.TrainRunner): same inputs, same Philox seed, no optimizer update -> identical loss and gradients."""
    from oracle.synth import config_for, synth_batch, synth_state_dict
    from sbgm_danra_b200 import score_sampling
    from sbgm_danra_b200._smoke import build_model
    from sbgm_danra_b200.score_unet import loss_fn, marginal_prob_std_fn
    cfg = config_for(n_lr=2, geo=True, seasons=True)
    net = build_model(cfg, synth_state_dict(cfg), "bf16x3", DEV).eval()     # eval: BatchNorm buffers do not move between steps
    b = synth_batch(batch=2, size=64, n_lr=2, geo=True, seasons=True)
    c = lambda v: None if v is None else v.to(DEV)
    snaps = []
    for step in range(5):
        score_sampling.manual_seed(3)
        net.zero_grad(set_to_none=True)
        loss = loss_fn(net, c(b.x), marginal_prob_std_fn, y=c(b.y), cond_img=c(b.cond_img), lsm_cond=c(b.lsm_cond),
                       topo_cond=c(b.topo_cond), sdf_cond=c(b.sdf_cond))
        loss.backward()
        snaps.append((loss.item(), {k: p.grad.clone() for k, p in net.named_parameters() if p.grad is not None}))
    runner = next(iter(net._train_runners.values()))
    assert runner.g_fwd is not None and runner.g_bwd is not None, "the step was never captured"
    for loss_k, grads_k in snaps[1:]:
        assert loss_k == snaps[0][0]
        assert grads_k.keys() == snaps[0][1].keys()
        for k in grads_k:
            assert torch.equal(grads_k[k], snaps[0][1][k]), k


def test_parameter_gradients_are_adopted_views_of_the_flat_buffer():
    """`.grad` tensors are views of the engine's flat gradient buffer (no per-parameter clone in AccumulateGrad); a `.grad`
    kept across a second backward (gradient accumulation) is detached first, so accumulation still adds."""
    from oracle.synth import config_for, synth_batch, synth_state_dict
    from sbgm_danra_b200 import score_sampling
    from sbgm_danra_b200._smoke import build_model
    from sbgm_danra_b200.score_unet import loss_fn, marginal_prob_std_fn
    cfg = config_for(n_lr=1)
    net = build_model(cfg, synth_state_dict(cfg), "bf16x3", DEV).eval()
    b = synth_batch(batch=2, size=32, n_lr=1)
    c = lambda v: None if v is None else v.to(DEV)

    def backward():
        score_sampling.manual_seed(3)
        loss_fn(net, c(b.x), marginal_prob_std_fn, cond_img=c(b.cond_img), sdf_cond=c(b.sdf_cond)).backward()

    for _ in range(4):                                  # eager steps, then the captured graphs
        net.zero_grad(set_to_none=True)
        backward()
        flat = next(iter(net._train_runners.values()))
        storages = {p.grad.untyped_storage().data_ptr() for p in net.parameters() if p.grad is not None}
        assert len(storages) == 1, "every gradient should live in one flat buffer"
    single = {k: p.grad.clone() for k, p in net.named_parameters() if p.grad is not None}
    backward()                                          # no zero_grad: accumulate on top of the adopted views
    for k, p in net.named_parameters():
        if p.grad is not None:
            assert torch.equal(p.grad, 2 * single[k]), k
    del flat


@pytest.mark.parametrize("precision", ["fp32", "bf16x3"])
def test_train_mode_batchnorm_forward_matches_reference_golden(golden, precision):
    """`.train()` forward under no_grad (the generation.py:47 quirk: sampling with batch statistics)."""
    from oracle.synth import config_for, synth_batch, synth_state_dict
    from sbgm_danra_b200._smoke import build_model
    cfg = config_for(n_lr=2, geo=True, seasons=True)
    net = build_model(cfg, synth_state_dict(cfg), precision, DEV).train()
    b = synth_batch(batch=2, size=64, n_lr=2, geo=True, seasons=True)
    with torch.no_grad():
        out = net(*[None if v is None else v.to(DEV) for v in b.model_args()]).cpu()
    err = rel_l2(out, golden["fwd_c3_64_cin7_seasons/score_bn_train"])
    print(f"train-mode BN forward [{precision}] rel-L2 = {err:.3e}")
    assert err < {"fp32": 1e-4, "bf16x3": 1e-3}[precision]


@pytest.mark.parametrize("precision", ["fp32", "bf16x3"])
def test_transpose_decoder_trains(precision):
    """`use_resize_conv=False` (ConvTranspose2d decoder, the reference's ablation switch): loss and all gradients against
    the oracle's autograd."""
    from oracle import philox_ref, score_ref
    from oracle.synth import config_for, synth_batch, synth_state_dict
    from sbgm_danra_b200 import score_sampling
    from sbgm_danra_b200._smoke import build_model
    from sbgm_danra_b200.score_unet import loss_fn, marginal_prob_std_fn
    cfg = config_for(n_lr=1, use_resize_conv=False, activation="gelu", n_heads=8)
    sd = synth_state_dict(cfg)
    # 64x64: at 32x32 the deepest BatchNorm layers normalise over batch x 1x1 = 4 values per channel in train mode, where a
    # 1e-5 perturbation (split-bf16 storage) flips ReLU masks -- measured 6 % gradient differences that are conditioning,
    # not arithmetic (every kernel involved passes its own test at 1e-5; eval-mode BatchNorm agrees to 4e-6)
    b = synth_batch(batch=4, size=64, n_lr=1)
    net = build_model(cfg, sd, precision, DEV).train()
    score_sampling.manual_seed(5)
    loss = loss_fn(net, b.x.to(DEV), marginal_prob_std_fn, cond_img=b.cond_img.to(DEV))
    loss.backward()
    sdo = {k: (v.clone().requires_grad_() if v.is_floating_point() and not k.endswith(("running_mean", "running_var", ".W")) else v.clone())
           for k, v in sd.items()}
    u = torch.from_numpy(philox_ref.uniform(4, 5, philox_ref.DRAW_DSM_T))
    z = torch.from_numpy(philox_ref.normal(b.x.numel(), 5, philox_ref.DRAW_DSM_Z)).reshape(b.x.shape)
    lo = score_ref.dsm_loss(sdo, cfg, b.x, u * (1.0 - 1e-3) + 1e-3, z, None, b.cond_img, None, None, None, bn_train=True)
    lo.backward()
    assert abs(loss.item() - lo.item()) / abs(lo.item()) < {"fp32": 1e-4, "bf16x3": 1e-3}[precision]
    params = dict(net.named_parameters())
    used = [k for k, v in sdo.items() if torch.is_tensor(v) and v.requires_grad and v.grad is not None]
    assert any("transpose.weight" in k for k in used)
    for k in used:
        assert params[k].grad is not None, k
        if "transpose" in k:
            assert rel_l2(params[k].grad.cpu(), sdo[k].grad) < {"fp32": 1e-3, "bf16x3": 2e-3}[precision], k
    whole = rel_l2(torch.cat([params[k].grad.cpu().reshape(-1) for k in used]), torch.cat([sdo[k].grad.reshape(-1) for k in used]))
    if os.environ.get("SBGM_TEST_VERBOSE"):
        for k in used:
            print(f"   {rel_l2(params[k].grad.cpu(), sdo[k].grad):.2e}  {k}")
    worst = sorted(((rel_l2(params[k].grad.cpu(), sdo[k].grad), k) for k in used), reverse=True)[:6]
    print(f"transpose decoder [{precision}]: loss {loss.item():.5f} vs {lo.item():.5f}, whole-gradient rel-L2 {whole:.2e}; worst {worst}")
    assert whole < {"fp32": 1e-4, "bf16x3": 1e-3}[precision]


def test_sampling_in_train_mode_uses_batch_statistics():
    """`model.train()` while sampling (generation.py:47 quirk): EM trajectory against the oracle sampler whose score uses
    BatchNorm batch statistics; the running statistics move, as they do in the reference."""
    from oracle import samplers_ref, score_ref
    from oracle.synth import config_for, synth_batch, synth_state_dict
    from sbgm_danra_b200 import score_sampling as ss
    from sbgm_danra_b200._smoke import build_model
    from sbgm_danra_b200.score_unet import diffusion_coeff_fn, marginal_prob_std_fn
    cfg = config_for(n_lr=1)
    sd = synth_state_dict(cfg)
    net = build_model(cfg, sd, "bf16x3", DEV).train()
    b = synth_batch(batch=4, size=32, n_lr=1, shared_cond=True)
    rm0 = net.encoder.bn1.running_mean.clone()
    ss.manual_seed(21)
    got = ss.Euler_Maruyama_sampler(net, marginal_prob_std_fn, diffusion_coeff_fn, batch_size=4, num_steps=5, device=DEV,
                                    img_size=32, cond_img=b.cond_img.to(DEV)).cpu()
    with torch.no_grad():
        want = samplers_ref.euler_maruyama(lambda x, t: score_ref.score_forward(sd, cfg, x, t, None, b.cond_img, bn_train=True),
                                           score_ref.marginal_prob_std, score_ref.diffusion_coeff, 4, 5, img_size=32,
                                           noise=samplers_ref.philox_noise(21))
    err = rel_l2(got, want)
    print(f"train-mode EM (5 steps) rel-L2 vs oracle = {err:.3e}")
    assert err < 2e-3
    assert not torch.equal(net.encoder.bn1.running_mean, rm0)
    # the step is ONE captured graph on the training engine's forward (score_sampling._TrainModeStep)
    plan = ss._PLAN_CACHE[0][1]
    assert isinstance(plan, ss._TrainModeStep) and plan.graph is not None
    nbt = int(net.encoder.bn1.num_batches_tracked)
    ss.manual_seed(21)              # a second call re-uses the plan; batch statistics do not depend on the running ones
    again = ss.Euler_Maruyama_sampler(net, marginal_prob_std_fn, diffusion_coeff_fn, batch_size=4, num_steps=5, device=DEV,
                                      img_size=32, cond_img=b.cond_img.to(DEV)).cpu()
    assert ss._PLAN_CACHE[0][1] is plan and torch.equal(again, got)
    assert int(net.encoder.bn1.num_batches_tracked) == nbt + 5          # one update per network evaluation, as torch counts them
    ss.clear_sampler_cache()


def test_train_mode_pc_sampling_with_labels_and_guidance_matches_oracle():
    """Predictor-corrector in `.train()` with season labels and classifier-free guidance: four batch-statistics evaluations
    per step (conditional + null branch for the corrector and for the predictor, each with its OWN batch statistics, as the
    reference's two separate forwards have -- never the 2B-wide form)."""
    from oracle import samplers_ref, score_ref
    from oracle.synth import config_for, synth_batch, synth_state_dict
    from sbgm_danra_b200 import score_sampling as ss
    from sbgm_danra_b200._smoke import build_model
    from sbgm_danra_b200.score_unet import diffusion_coeff_fn, marginal_prob_std_fn
    ck = dict(n_lr=2, geo=True, seasons=True)
    cfg = config_for(**ck)
    sd = synth_state_dict(cfg)
    net = build_model(cfg, sd, "bf16x3", DEV).train()
    b = synth_batch(batch=4, size=32, shared_cond=True, **ck)
    guid = {"classifier_free_guidance": {"enabled": True, "guidance_scale": 1.5}}
    c = lambda v: v.to(DEV)
    ss.manual_seed(5)
    got = ss.pc_sampler(net, marginal_prob_std_fn, diffusion_coeff_fn, batch_size=4, num_steps=3, snr=0.16, device=DEV, img_size=32,
                        y=c(b.y), cond_img=c(b.cond_img), lsm_cond=c(b.lsm_cond), topo_cond=c(b.topo_cond), cfg=guid).cpu()
    model = lambda *a: score_ref.score_forward(sd, cfg, *a, bn_train=True)
    score = lambda x, t: samplers_ref.guided_score(model, x, t, b.y, b.cond_img, b.lsm_cond, b.topo_cond, scale=1.5)
    with torch.no_grad():
        want = samplers_ref.predictor_corrector(score, score_ref.marginal_prob_std, score_ref.diffusion_coeff, 4, 3, img_size=32,
                                                noise=samplers_ref.philox_noise(5))
    err = rel_l2(got, want)
    print(f"train-mode guided PC (3 steps) rel-L2 vs oracle = {err:.3e}")
    assert err < 2e-3 and isinstance(ss._PLAN_CACHE[0][1], ss._TrainModeStep)
    ss.clear_sampler_cache()


@pytest.mark.parametrize("prec", ["fp32", "bf16x3", "bf16"])
@pytest.mark.parametrize("shape", [(4, 512, 1, 1), (2, 64, 16, 16), (3, 128, 8, 4), (4, 256, 2, 2)])
def test_conv_transpose_layer_forward_backward(E, T, prec, shape):
    """ConvTranspose2d(c, c, 2, 2) of the use_resize_conv=False decoder: forward, input / weight / bias gradients."""
    fmt = FMTS[prec]
    n, c, h, w = shape
    wt = gen(c, c, 2, 2, seed=1, scale=c ** -0.5)
    bt = gen(c, seed=2, scale=0.1)
    x = stored(E, gen(n, c, h, w, seed=3), fmt).requires_grad_()
    dy = stored(E, gen(n, c, 2 * h, 2 * w, seed=4), fmt)
    wr, br = wt.clone().requires_grad_(), bt.clone().requires_grad_()
    want = F.conv_transpose2d(x, wr, br, stride=2)
    want.backward(dy)
    tk, grads = make_tk(T, fmt)
    layer = T.ConvTLayer("w", wt.to(DEV), bt.to(DEV), fmt, "b")
    xa = act_of(E, x.detach(), fmt)
    ya = tk.conv_transpose2x(xa, layer)
    tol = {"fp32": 2e-5, "bf16x3": 1e-4, "bf16": 2e-2}[prec]
    assert rel_l2(ya.to_nchw().cpu(), want.detach()) < tol
    tk.tape.add(ya, act_of(E, dy, fmt))
    run_tape(tk)
    e_dx = rel_l2(tk.tape.grads[xa.buf.data_ptr()].to_nchw().cpu(), x.grad)
    e_dw, e_db = rel_l2(grads["w"].cpu(), wr.grad), rel_l2(grads["b"].cpu(), br.grad)
    print(f"convT {shape} [{prec}] dx {e_dx:.2e} dW {e_dw:.2e} db {e_db:.2e}")
    assert e_dx < tol and e_dw < tol and e_db < tol


def test_gradient_accumulation_and_loss_scaling_in_graph_mode():
    """Two backward passes without zero_grad accumulate (the captured backward writes into a static flat buffer: param.grad
    must never alias it), and d(k * loss) = k * d(loss) (the grad_loss scalar reaches the loss-backward kernel)."""
    from oracle.synth import config_for, synth_batch, synth_state_dict
    from sbgm_danra_b200 import score_sampling
    from sbgm_danra_b200._smoke import build_model
    from sbgm_danra_b200.score_unet import loss_fn, marginal_prob_std_fn
    cfg = config_for(n_lr=1)
    net = build_model(cfg, synth_state_dict(cfg), "bf16x3", DEV).eval()
    b = synth_batch(batch=2, size=32, n_lr=1)

    def step(scale=1.0):
        score_sampling.manual_seed(9)
        loss = loss_fn(net, b.x.to(DEV), marginal_prob_std_fn, cond_img=b.cond_img.to(DEV))
        (loss * scale).backward()

    for _ in range(3):                      # eager, eager, capture + replay
        net.zero_grad(set_to_none=True)
        step()
    runner = next(iter(net._train_runners.values()))
    assert runner.g_bwd is not None
    net.zero_grad(set_to_none=True)
    step()
    single = {k: p.grad.clone() for k, p in net.named_parameters() if p.grad is not None}
    step()                                   # accumulates
    for k, p in net.named_parameters():
        if p.grad is not None:
            assert torch.allclose(p.grad, 2.0 * single[k], rtol=1e-6, atol=0.0), k
    net.zero_grad(set_to_none=True)
    step(scale=4.0)                          # a power of two commutes with every rounding on the path: exact
    for k, p in net.named_parameters():
        if p.grad is not None:
            assert torch.equal(p.grad, 4.0 * single[k]), k


def test_training_step_on_ragged_maps_96x96():
    """96x96 input: feature maps 48 / 24 / 12 / 6 / 3 -- pixel tiles with tails in the tensor-core weight gradient, odd sizes in
    the parity-sliced data gradients of the strided convolutions, attention over 36 and 9 tokens.  Eval-mode BatchNorm keeps the
    comparison well conditioned (see test_transpose_decoder_trains)."""
    from oracle import philox_ref, score_ref
    from oracle.synth import config_for, synth_batch, synth_state_dict
    from sbgm_danra_b200 import score_sampling
    from sbgm_danra_b200._smoke import build_model
    from sbgm_danra_b200.score_unet import loss_fn, marginal_prob_std_fn
    cfg = config_for(n_lr=1)
    sd = synth_state_dict(cfg)
    b = synth_batch(batch=2, size=96, n_lr=1)
    net = build_model(cfg, sd, "bf16x3", DEV).eval()
    score_sampling.manual_seed(17)
    loss = loss_fn(net, b.x.to(DEV), marginal_prob_std_fn, cond_img=b.cond_img.to(DEV), sdf_cond=b.sdf_cond.to(DEV))
    loss.backward()
    sdo = {k: (v.clone().requires_grad_() if v.is_floating_point() and not k.endswith(("running_mean", "running_var", ".W")) else v.clone())
           for k, v in sd.items()}
    u = torch.from_numpy(philox_ref.uniform(2, 17, philox_ref.DRAW_DSM_T))
    z = torch.from_numpy(philox_ref.normal(b.x.numel(), 17, philox_ref.DRAW_DSM_Z)).reshape(b.x.shape)
    lo = score_ref.dsm_loss(sdo, cfg, b.x, u * (1.0 - 1e-3) + 1e-3, z, None, b.cond_img, None, None, b.sdf_cond, bn_train=False)
    lo.backward()
    params = dict(net.named_parameters())
    used = [k for k, v in sdo.items() if torch.is_tensor(v) and v.requires_grad and v.grad is not None]
    whole = rel_l2(torch.cat([params[k].grad.cpu().reshape(-1) for k in used]), torch.cat([sdo[k].grad.reshape(-1) for k in used]))
    worst = max((rel_l2(params[k].grad.cpu(), sdo[k].grad), k) for k in used)
    print(f"96x96 training step: loss {loss.item():.4f} vs {lo.item():.4f}; whole-gradient rel-L2 {whole:.2e}; worst {worst}")
    assert abs(loss.item() - lo.item()) / abs(lo.item()) < 1e-3
    assert whole < 1e-3 and worst[0] < 5e-3


def test_reference_epoch_flow_train_validate_generate():
    """One epoch as the reference's L2 drives it (sbgm/training.py), twice over:
    `train_batches` (:246-422 -- dataset dict -> extract_samples -> zero_grad -> loss_fn -> backward INSIDE
    `torch.autograd.detect_anomaly(True)` -> optimizer.step -> .item()), `validate_batches` (:510-580 -- .eval(), loss_fn
    under `torch.inference_mode()`), then the sampler call of `generate_and_plot_samples` (:683-695 -- keyword arguments,
    `.squeeze().detach().cpu()`).  The second epoch re-uses whatever the first one cached (engines first built under
    inference mode are then used outside it)."""
    from oracle.synth import config_for, synth_batch, synth_state_dict
    from sbgm_danra_b200 import score_sampling
    from sbgm_danra_b200._smoke import build_model
    from sbgm_danra_b200.score_unet import diffusion_coeff_fn, loss_fn, marginal_prob_std_fn
    cfg = config_for(n_lr=2, geo=True, seasons=True)
    net = build_model(cfg, synth_state_dict(cfg), "bf16x3", DEV)
    b = synth_batch(batch=4, size=32, n_lr=2, geo=True, seasons=True)
    samples = {"temp_hr": b.x, "classifier": b.y, "prcp_lr": b.cond_img[:, :1], "temp_lr": b.cond_img[:, 1:],
               "lsm": b.lsm_cond, "topo": b.topo_cond, "sdf": b.sdf_cond}

    def extract(s):       # utils.extract_samples :405-480 (LR keys sorted and concatenated, everything .to(device).float())
        f = lambda v: v.to(DEV, non_blocking=True).float()
        lr = torch.cat([f(s[k]) for k in sorted(k for k in s if k.endswith("_lr"))], dim=1)
        return f(s["temp_hr"]), s["classifier"].to(DEV, non_blocking=True), lr, f(s["lsm"]), f(s["sdf"]), f(s["topo"])

    opt = torch.optim.Adam(net.parameters(), lr=1e-4)
    score_sampling.manual_seed(5)
    train_losses, val_losses = [], []
    for epoch in range(2):
        net.train()
        for _ in range(3):
            x, seasons, cond, lsm, sdf, topo = extract(samples)
            opt.zero_grad()
            batch_loss = loss_fn(net, x, marginal_prob_std_fn, y=seasons, cond_img=cond, lsm_cond=lsm, topo_cond=topo, sdf_cond=sdf)
            with torch.autograd.detect_anomaly(True):
                batch_loss.backward()
            opt.step()
            train_losses.append(batch_loss.item())
        net.eval()
        with torch.inference_mode():
            x, seasons, cond, lsm, sdf, topo = extract(samples)
            val_losses.append(loss_fn(net, x, marginal_prob_std_fn, y=seasons, cond_img=cond, lsm_cond=lsm, topo_cond=topo,
                                      sdf_cond=sdf).item())
        x, seasons, cond, lsm, sdf, topo = extract(samples)
        for sampler in (score_sampling.pc_sampler, score_sampling.Euler_Maruyama_sampler):
            gen = sampler(score_model=net, marginal_prob_std=marginal_prob_std_fn, diffusion_coeff=diffusion_coeff_fn,
                          batch_size=4, num_steps=3, device=DEV, img_size=32, y=seasons, cond_img=cond, lsm_cond=lsm,
                          topo_cond=topo)
            gen = gen.squeeze().detach().cpu()
            assert gen.shape == (4, 32, 32) and torch.isfinite(gen).all()
    assert all(np.isfinite(train_losses)) and all(np.isfinite(val_losses)), (train_losses, val_losses)
    grads = [p.grad for p in net.parameters() if p.grad is not None]
    assert len(grads) > 100 and all(torch.isfinite(g).all() for g in grads)


# ---- optimizer ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,wd", [("Adam", 0.0), ("Adam", 0.05), ("AdamW", 0.05)])
def test_one_launch_adam_matches_torch(kind, wd):
    """sbgm_danra_b200.optim.Adam / AdamW (one kernel over all tensors) against torch.optim's, same gradients, 5 steps; the state
    dict of one loads into the other (the reference checkpoints 'optimizer_params', training.py:241)."""
    from sbgm_danra_b200 import optim
    gen_ = torch.Generator().manual_seed(0)
    shapes = [(64, 7, 8, 8), (4097,), (1,), (512, 512, 3, 3), (3, 5)]
    base = [torch.randn(s, generator=gen_) for s in shapes]
    flat = torch.zeros(sum(t.numel() for t in base) + 3, device=DEV)          # an UNALIGNED view too (scalar path of the kernel)
    mine = [torch.nn.Parameter(t.clone().to(DEV)) for t in base]
    odd = torch.nn.Parameter(flat[3:3 + 77])
    theirs = [torch.nn.Parameter(t.clone().to(DEV)) for t in base] + [torch.nn.Parameter(torch.zeros(77, device=DEV))]
    mine.append(odd)
    a = getattr(optim, kind)(mine, lr=3e-3, weight_decay=wd)
    b = getattr(torch.optim, kind)(theirs, lr=3e-3, weight_decay=wd)
    for step in range(5):
        for p, q in zip(mine, theirs):
            g = torch.randn(p.shape, generator=gen_).to(DEV) * (10.0 ** (step - 2))
            p.grad, q.grad = g.clone(), g.clone()
        a.step()
        b.step()
    for p, q in zip(mine, theirs):
        assert torch.allclose(p, q, rtol=2e-6, atol=1e-7), float((p - q).abs().max())
    # state dicts are interchangeable
    sa, sb = a.state_dict(), b.state_dict()
    assert sa["param_groups"][0].keys() == sb["param_groups"][0].keys()
    assert float(sa["state"][0]["step"]) == float(sb["state"][0]["step"]) == 5.0
    assert torch.allclose(sa["state"][3]["exp_avg_sq"], sb["state"][3]["exp_avg_sq"], rtol=2e-6, atol=1e-12)
    b.load_state_dict(sa)
    a.load_state_dict(sb)
    for p, q in zip(mine, theirs):
        g = torch.ones_like(p)
        p.grad, q.grad = g, g.clone()
    a.step()
    b.step()
    for p, q in zip(mine, theirs):
        assert torch.allclose(p, q, rtol=4e-6, atol=1e-7)


@pytest.mark.parametrize("prec", ["fp32", "bf16x3", "bf16"])
@pytest.mark.parametrize("n,hw,c,per_sample", [(1, 300, 768, False),       # one block per channel vector (Linear bias gradients)
                                               (3, 4096, 128, False),      # same, 512 threads
                                               (4, 128 * 96, 64, False),   # > 32768 pixels: ticketed last-block reduction, twice on one scratch
                                               (3, 1000, 64, True)])       # per-sample sums + total (time-projection gradients)
def test_channel_sums(E, prec, n, hw, c, per_sample):
    from sbgm_danra_b200 import _lib
    from sbgm_danra_b200._lib import call
    fmt = FMTS[prec]
    x = stored(E, gen(n, c, 1, hw, seed=1), fmt)
    xa = act_of(E, x, fmt)
    ws = torch.zeros(_lib.query("sbgm_channel_sums_scratch_floats", n, c), device=DEV)
    tot = torch.zeros(c, device=DEV)
    per = torch.zeros(n, c + 5, device=DEV) if per_sample else None
    st = torch.cuda.current_stream().cuda_stream
    for _ in range(2):
        call("sbgm_channel_sums", xa.ptr, xa.plane, fmt, n, hw, c, None if per is None else per.data_ptr(), c + 5, tot.data_ptr(),
             ws.data_ptr(), st)
    want = x.double().sum(dim=(2, 3))
    assert rel_l2(tot.cpu().double(), want.sum(0)) < 1e-5
    if per_sample:
        assert rel_l2(per[:, :c].cpu().double(), want) < 1e-5
    assert int(ws[:4096].view(torch.int32).abs().sum()) == 0


def test_graph_capture_survives_a_pinning_thread():
    """The training graphs are captured on the third step, while a DataLoader(pin_memory=True) thread may be allocating pinned
    memory and querying events: the capture must not be invalidated by CUDA calls of OTHER threads (capture_error_mode)."""
    import threading
    from oracle.synth import config_for, synth_batch, synth_state_dict
    from sbgm_danra_b200 import score_sampling
    from sbgm_danra_b200._smoke import build_model
    from sbgm_danra_b200.score_unet import loss_fn, marginal_prob_std_fn
    cfg = config_for(n_lr=1)
    net = build_model(cfg, synth_state_dict(cfg), "bf16", DEV).eval()
    b = synth_batch(batch=2, size=32, n_lr=1)
    stop = threading.Event()

    def pin_loop():
        while not stop.is_set():
            buf = torch.empty(1 << 16, dtype=torch.uint8, pin_memory=True)     # cudaHostAlloc: "unsafe" during a global-mode capture
            ev = torch.cuda.Event()
            ev.query()
            del buf

    th = threading.Thread(target=pin_loop, daemon=True)
    th.start()
    try:
        losses = []
        for _ in range(5):
            score_sampling.manual_seed(5)
            net.zero_grad(set_to_none=True)
            loss = loss_fn(net, b.x.to(DEV), marginal_prob_std_fn, cond_img=b.cond_img.to(DEV))
            loss.backward()
            losses.append(float(loss))
    finally:
        stop.set()
        th.join()
    assert all(abs(v - losses[0]) <= 1e-6 * abs(losses[0]) for v in losses), losses


def test_failed_graph_capture_falls_back_to_eager_and_is_retried(monkeypatch):
    """A capture that is invalidated (here: a synchronize inside it, once) must cost one eager step, not the training run: the step
    still returns the right loss and gradients, and the next step captures."""
    import warnings
    from oracle.synth import config_for, synth_batch, synth_state_dict
    from sbgm_danra_b200 import score_sampling, train_engine
    from sbgm_danra_b200._smoke import build_model
    from sbgm_danra_b200.score_unet import loss_fn, marginal_prob_std_fn
    cfg = config_for(n_lr=1)
    net = build_model(cfg, synth_state_dict(cfg), "bf16", DEV).eval()
    b = synth_batch(batch=2, size=32, n_lr=1)
    orig_pack = train_engine.TrainEngine._pack
    fired = []

    def pack_once_broken(self):
        if torch.cuda.is_current_stream_capturing() and not fired:
            fired.append(1)
            torch.cuda.synchronize()            # illegal inside a capture: invalidates it and raises
        return orig_pack(self)

    monkeypatch.setattr(train_engine.TrainEngine, "_pack", pack_once_broken)
    snaps = []
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always")
        for _ in range(6):
            score_sampling.manual_seed(11)
            net.zero_grad(set_to_none=True)
            loss = loss_fn(net, b.x.to(DEV), marginal_prob_std_fn, cond_img=b.cond_img.to(DEV))
            loss.backward()
            snaps.append((float(loss), torch.cat([p.grad.flatten() for p in net.parameters() if p.grad is not None]).clone()))
    assert fired and any("capture" in str(w.message) for w in caught)
    for lo, g in snaps[1:]:
        assert lo == snaps[0][0] and torch.equal(g, snaps[0][1])
    (runner,) = net.__dict__["_train_runners"].values()
    assert runner.g_fwd is not None and runner.capture_failures == 1 and runner.use_graphs


def test_failed_backward_capture_redoes_the_step_eagerly(monkeypatch):
    """The forward graph has already run when the backward capture fails: the step is redone on the eager launch sequence from the
    static inputs (same loss, same gradients, bit for bit), both graphs are dropped and captured again on the next step."""
    import warnings
    from oracle.synth import config_for, synth_batch, synth_state_dict
    from sbgm_danra_b200 import score_sampling, train_engine
    from sbgm_danra_b200._smoke import build_model
    from sbgm_danra_b200.score_unet import loss_fn, marginal_prob_std_fn
    cfg = config_for(n_lr=1)
    net = build_model(cfg, synth_state_dict(cfg), "bf16", DEV).eval()
    b = synth_batch(batch=2, size=32, n_lr=1)
    orig_backward = train_engine.TrainEngine.backward
    fired = []

    def backward_once_broken(self, dscore):
        if torch.cuda.is_current_stream_capturing() and not fired:
            fired.append(1)
            torch.cuda.synchronize()            # illegal inside a capture: invalidates it and raises
        return orig_backward(self, dscore)

    monkeypatch.setattr(train_engine.TrainEngine, "backward", backward_once_broken)
    snaps = []
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always")
        for _ in range(6):
            score_sampling.manual_seed(11)
            net.zero_grad(set_to_none=True)
            loss = loss_fn(net, b.x.to(DEV), marginal_prob_std_fn, cond_img=b.cond_img.to(DEV))
            loss.backward()
            snaps.append((float(loss), torch.cat([p.grad.flatten() for p in net.parameters() if p.grad is not None]).clone()))
    assert fired and any("capture" in str(w.message) for w in caught)
    for lo, g in snaps[1:]:
        assert lo == snaps[0][0] and torch.equal(g, snaps[0][1])
    (runner,) = net.__dict__["_train_runners"].values()
    assert runner.g_fwd is not None and runner.g_bwd is not None and runner.capture_failures == 1 and not runner.busy


def test_dead_cycle_owning_a_cuda_graph_does_not_break_the_next_capture():
    """The root cause of the order-dependent capture failure: an unreachable reference cycle that owns a CUDA graph (an earlier
    model and its runner) is finalised by the cyclic collector at an arbitrary allocation -- inside a capture that is "not
    permitted" and invalidates it.  graph_capture collects before the capture and pauses the collector during it."""
    import gc
    from oracle.synth import config_for, synth_batch, synth_state_dict
    from sbgm_danra_b200 import score_sampling
    from sbgm_danra_b200._smoke import build_model
    from sbgm_danra_b200.score_unet import loss_fn, marginal_prob_std_fn

    class Holder:
        pass

    gc.collect()
    g = torch.cuda.CUDAGraph()
    buf = torch.zeros(1024, device=DEV)
    with torch.cuda.graph(g):
        buf += 1
    a, b_ = Holder(), Holder()
    a.other, b_.other, a.graph = b_, a, g          # a cycle that owns the graph ...
    for _ in range(3):
        gc.collect()                               # ... promoted to the oldest generation while alive ...
    del a, b_, g                                   # ... and now dead, waiting for a full collection
    gc.set_threshold(50, 2, 2)                     # make full collections frequent for the rest of this test
    try:
        cfg = config_for(n_lr=1)
        net = build_model(cfg, synth_state_dict(cfg), "bf16", DEV).eval()
        b = synth_batch(batch=2, size=32, n_lr=1)
        for _ in range(4):
            score_sampling.manual_seed(2)
            net.zero_grad(set_to_none=True)
            loss_fn(net, b.x.to(DEV), marginal_prob_std_fn, cond_img=b.cond_img.to(DEV)).backward()
        (runner,) = net.__dict__["_train_runners"].values()
        assert runner.g_fwd is not None and runner.g_bwd is not None and getattr(runner, "capture_failures", 0) == 0
    finally:
        gc.set_threshold(700, 10, 10)
