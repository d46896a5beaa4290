"""GPU parity tests, one per C-ABI kernel: each calls the CUDA path through the C ABI (ctypes) and
compares with a plain torch fp32 CPU evaluation of the same operator on the same seeded inputs.

Tolerances (relative L2 unless noted): fp32 kernels 1e-5; bf16x3 (split-bf16 tensor-core) 1e-4;
bf16 2e-2 -- written next to each check."""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import rel_l2

pytestmark = pytest.mark.gpu

FMTS = {"fp32": 0, "bf16": 1, "bf16x3": 2, "fp16x2": 3}
# fp16x2: float16 activations (2^-12 relative rounding on load and on store), weights exact to 22 bits
TOL = {"fp32": 2e-5, "bf16": 2e-2, "bf16x3": 1e-4, "fp16x2": 6e-4}
ELEM_TOL = {"fp32": 1e-6, "bf16": 6e-3, "bf16x3": 2e-5, "fp16x2": 4e-4}   # storage round-trip only


@pytest.fixture(scope="module")
def E():
    from sbgm_danra_b200 import engine
    return engine


def gen(*shape, seed=0, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(*shape, generator=g) * scale


def act_of(E, x, fmt):
    return E.Act.from_nchw(x.cuda(), fmt)


@pytest.mark.parametrize("prec", list(FMTS))
def test_layout_roundtrip(E, prec):
    x = gen(3, 72, 5, 7)
    y = act_of(E, x, FMTS[prec]).to_nchw().cpu()
    assert rel_l2(y, x) < ELEM_TOL[prec]


@pytest.mark.parametrize("rows,labels", [(5, False), (3, True)])
def test_time_embed_project(E, rows, labels):
    from oracle import score_ref
    te = 256
    tp = E.TimeProjector(torch.device("cuda"), te)
    W0, W1 = gen(128, seed=1, scale=30.0), gen(128, seed=2, scale=30.0)
    s0, s1 = tp.add_set(W0.cuda()), tp.add_set(W1.cuda())
    heads = [("a", s0, 64), ("b", s0, 128), ("c", s1, 256)]
    ws = {}
    for i, (name, s, c) in enumerate(heads):
        ws[name] = (gen(c, te, seed=10 + i, scale=0.06), gen(c, seed=20 + i, scale=0.1))
        tp.add_head(name, s, ws[name][0].cuda(), ws[name][1].cuda())
    lab = gen(5, te, seed=30, scale=0.5)
    tp.label_emb = lab.cuda() if labels else None
    tp.finalize()
    t = torch.rand(rows, generator=torch.Generator().manual_seed(3))
    y = torch.tensor([1, 4, 0][:rows]) if labels else None
    out = tp(t.cuda(), None if y is None else y.cuda()).cpu()
    for name, s, c in heads:
        emb = score_ref.fourier_embed(W0 if s == s0 else W1, t)
        if labels and s == s0:
            emb = emb + lab[y]
        want = F.linear(F.silu(emb), *ws[name])
        got = tp.cols(out, name)
        assert rel_l2(got, want) < 2e-5, name


@pytest.mark.parametrize("prec", ["fp32", "bf16x3"])
@pytest.mark.parametrize("cc,bcast", [(1, False), (6, True)])
def test_stem_conv(E, prec, cc, bcast):
    from sbgm_danra_b200._lib import call
    n, h = 3, 64
    x = gen(n, 1, h, h, seed=1)
    planes = gen(1 if bcast else n, cc, h, h, seed=2)
    w = gen(64, cc + 1, 8, 8, seed=3, scale=0.1)
    tproj = gen(n, 100, seed=4)
    full = torch.cat([x, planes.expand(n, -1, -1, -1)], 1)
    want = F.conv2d(full, w, stride=2, padding=3) + tproj[:, 10:74, None, None]
    wp = w.permute(1, 2, 3, 0).reshape(cc + 1, 64, 64).contiguous().cuda()
    fmt = FMTS[prec]
    xd, pd, td = x.cuda(), planes.cuda().contiguous(), tproj.cuda()
    tview = td[:, 10:74]
    st = torch.cuda.current_stream().cuda_stream
    # (a) everything in one launch
    out = E.Act(fmt, n, h // 2, h // 2, 64, "cuda")
    call("sbgm_stem_conv", xd.data_ptr(), pd.data_ptr(), pd.shape[0], cc, 0, cc + 1, wp.data_ptr(), None, 0,
         tview.data_ptr(), tview.stride(0), out.ptr, out.plane, fmt, n, h, h, st)
    assert rel_l2(out.to_nchw().cpu(), want) < TOL[prec]
    # (b) step-invariant conditioning partial + per-step x channel (sampler split)
    part = E.Act(0, pd.shape[0], h // 2, h // 2, 64, "cuda")
    call("sbgm_stem_conv", None, pd.data_ptr(), pd.shape[0], cc, 1, cc + 1, wp.data_ptr(), None, 0, None, 0,
         part.ptr, part.plane, 0, pd.shape[0], h, h, st)
    out2 = E.Act(fmt, n, h // 2, h // 2, 64, "cuda")
    call("sbgm_stem_conv", xd.data_ptr(), None, 1, cc, 0, 1, wp.data_ptr(), part.ptr, pd.shape[0],
         tview.data_ptr(), tview.stride(0), out2.ptr, out2.plane, fmt, n, h, h, st)
    assert rel_l2(out2.to_nchw().cpu(), want) < TOL[prec]


CONV_CASES = [
    # n, h, w, cin, cout, k, stride, pad, epilogue
    (2, 32, 32, 64, 64, 3, 1, 1, "plain"),
    (2, 32, 32, 64, 64, 3, 1, 1, "full"),
    (3, 8, 8, 128, 256, 3, 1, 1, "full"),
    (2, 16, 16, 64, 128, 3, 2, 1, "relu"),
    (2, 16, 16, 64, 128, 1, 2, 0, "plain"),
    (2, 32, 32, 64, 64, 8, 2, 3, "relu"),
    (3, 4, 4, 256, 512, 3, 1, 1, "full"),
    (5, 2, 2, 512, 512, 3, 1, 1, "plain"),
    (3, 1, 1, 512, 512, 3, 1, 1, "plain"),
    (1, 1, 200, 128, 384, 1, 1, 0, "gelu"),       # Linear over 200 tokens (tail masking)
    (1, 1, 1024, 512, 1536, 1, 1, 0, "plain"),    # in_proj of the 512-channel attention
    (1, 64, 64, 64, 64, 3, 1, 1, "full"),
    (3, 8, 16, 64, 64, 3, 1, 1, "full"),          # single tile per image of the persistent 64->64 kernel
    (70, 16, 32, 64, 64, 3, 1, 1, "relu"),        # 280 tiles: more than one wave of the persistent kernel
    (2, 12, 24, 64, 192, 3, 1, 1, "full"),        # non power-of-two spatial, cout = 3 x 64
    # halo-slab mode of the generic kernel (3x3, stride 1, maps tileable by 16 rows x 8 columns)
    (3, 32, 32, 128, 128, 3, 1, 1, "full"),
    (2, 16, 16, 256, 256, 3, 1, 1, "relu"),
    (2, 16, 24, 128, 64, 3, 1, 1, "plain"),       # 64-wide tile, three tiles per row
    (2, 32, 8, 192, 320, 3, 1, 1, "full"),        # odd number of channel blocks (slab ring parity), cout = 5 x 64
    (40, 16, 16, 128, 256, 3, 1, 1, "gelu"),      # several waves
    (64, 8, 8, 256, 256, 3, 1, 1, "full"),        # 8 x 8 maps: tiles of two images, permuted tensor maps
    (5, 8, 8, 512, 512, 3, 1, 1, "full"),         # same with an odd image count and split-K over channel blocks
    (3, 24, 8, 128, 128, 3, 1, 1, "relu"),        # 24 rows: 8-row tiles
    (33, 8, 16, 192, 64, 3, 1, 1, "plain"),
    # weight multicast over a CTA pair (slab mode, cin / cout >= 512, single-plane formats): two-image tiles, and an ODD number
    # of pixel tiles (the pair's second CTA of the last cluster has no tile)
    (64, 8, 8, 512, 512, 3, 1, 1, "full"),
    (19, 16, 8, 512, 512, 3, 1, 1, "relu"),
]


@pytest.mark.parametrize("prec", list(FMTS))
@pytest.mark.parametrize("case", CONV_CASES, ids=lambda c: "x".join(map(str, c)))
def test_conv2d(E, prec, case):
    n, h, w, cin, cout, k, stride, pad, epi = case
    fmt = FMTS[prec]
    x = gen(n, cin, h, w, seed=1)
    wt = gen(cout, cin, k, k, seed=2, scale=1.0 / math.sqrt(cin * k * k))
    bias = gen(cout, seed=3, scale=0.1) if epi != "plain" else None
    ho, wo = (h + 2 * pad - k) // stride + 1, (w + 2 * pad - k) // stride + 1
    res = gen(n, cout, ho, wo, seed=4) if epi == "full" else None
    tproj = gen(n, cout + 16, seed=5) if epi == "full" else None
    act = {"plain": 0, "full": 1, "relu": 1, "gelu": 3}[epi]
    want = F.conv2d(x, wt, bias, stride=stride, padding=pad)
    if res is not None:
        want = want + res
    want = {0: lambda v: v, 1: F.relu, 3: F.gelu}[act](want)
    if tproj is not None:
        want = want + tproj[:, 8:8 + cout, None, None]   # 16-byte aligned column offset (ABI requirement)
    kern = E.Kernels(fmt, torch.device("cuda"))
    sd = {"w": wt}
    if bias is not None:
        sd["b"] = bias
    cw = E._Packer(sd, fmt, torch.device("cuda")).conv("w", "b" if bias is not None else None)
    tp = tproj.cuda()[:, 8:8 + cout] if tproj is not None else None
    out = kern.conv(act_of(E, x, fmt), cw, stride=stride, pad=pad, act=act,
                    residual=None if res is None else act_of(E, res, fmt), tproj=tp)
    torch.cuda.synchronize()
    assert (out.h, out.w, out.c) == (ho, wo, cout)
    err = rel_l2(out.to_nchw().cpu(), want)
    assert err < TOL[prec], f"rel-L2 {err:.3e}"


def test_conv_bn_fold(E):
    """Eval-mode BatchNorm folded into the packed convolution (engine._Packer.conv)."""
    x = gen(2, 64, 16, 16, seed=1)
    sd = {"c.weight": gen(128, 64, 3, 3, seed=2, scale=0.05), "bn.weight": 1 + 0.1 * gen(128, seed=3),
          "bn.bias": gen(128, seed=4, scale=0.1), "bn.running_mean": gen(128, seed=5, scale=0.1),
          "bn.running_var": torch.rand(128, generator=torch.Generator().manual_seed(6)) + 0.5}
    want = F.relu(F.batch_norm(F.conv2d(x, sd["c.weight"], padding=1), sd["bn.running_mean"], sd["bn.running_var"],
                               sd["bn.weight"], sd["bn.bias"], False, 0.0, 1e-5))
    for prec in ("fp32", "bf16x3"):
        fmt = FMTS[prec]
        cw = E._Packer(sd, fmt, torch.device("cuda")).conv("c.weight", bn="bn")
        out = E.Kernels(fmt, torch.device("cuda")).conv(act_of(E, x, fmt), cw, pad=1, act=1)
        assert rel_l2(out.to_nchw().cpu(), want) < TOL[prec]


@pytest.mark.parametrize("prec", list(FMTS))
@pytest.mark.parametrize("c,groups,hw,fused", [(64, 8, 32, True), (512, 8, 8, False), (128, 128, 16, True), (256, 8, 4, True)])
def test_groupnorm(E, prec, c, groups, hw, fused):
    fmt = FMTS[prec]
    n = 3
    x = gen(n, c, hw, hw, seed=1) * 2 + 0.5
    instance = groups == c
    gamma = None if instance else 1 + 0.2 * gen(c, seed=2)
    beta = None if instance else gen(c, seed=3, scale=0.2)
    skip = gen(n, c, hw, hw, seed=4) if fused else None
    tproj = gen(n, c, seed=5) if fused else None
    if prec != "fp32":   # compare against the norm of what the kernel actually reads
        x = act_of(E, x, fmt).to_nchw().cpu()
    want = F.instance_norm(x, eps=1e-5) if instance else F.group_norm(x, groups, gamma, beta, 1e-5)
    if fused:
        want = F.silu(want + skip + tproj[:, :, None, None])
    kern = E.Kernels(fmt, torch.device("cuda"))
    out = kern.groupnorm(act_of(E, x, fmt), None if gamma is None else gamma.cuda(), None if beta is None else beta.cuda(),
                         groups, act=2 if fused else 0, skip=None if skip is None else act_of(E, skip, fmt),
                         tproj=None if tproj is None else tproj.cuda())
    tol = {"fp32": 1e-5, "bf16x3": 3e-5, "bf16": 8e-3, "fp16x2": 5e-4}[prec]
    assert rel_l2(out.to_nchw().cpu(), want) < tol


@pytest.mark.parametrize("prec", list(FMTS))
@pytest.mark.parametrize("c", [128, 256, 512])
def test_layernorm(E, prec, c):
    fmt = FMTS[prec]
    x = gen(1, c, 1, 77, seed=1) * 3 + 1
    if prec != "fp32":
        x = act_of(E, x, fmt).to_nchw().cpu()
    g, b = 1 + 0.2 * gen(c, seed=2), gen(c, seed=3, scale=0.2)
    want = F.layer_norm(x[0, :, 0].T, (c,), g, b, 1e-5).T[None, :, None]
    out = E.Kernels(fmt, torch.device("cuda")).layernorm(act_of(E, x, fmt), g.cuda(), b.cuda())
    tol = {"fp32": 1e-5, "bf16x3": 3e-5, "bf16": 8e-3, "fp16x2": 5e-4}[prec]
    assert rel_l2(out.to_nchw().cpu(), want) < tol


@pytest.mark.parametrize("prec", list(FMTS))
def test_upsample2x(E, prec):
    fmt = FMTS[prec]
    x = gen(2, 64, 5, 9, seed=1)
    if prec != "fp32":
        x = act_of(E, x, fmt).to_nchw().cpu()
    want = F.interpolate(x, scale_factor=2, mode="bilinear", align_corners=False)
    out = E.Kernels(fmt, torch.device("cuda")).upsample2x(act_of(E, x, fmt))
    assert rel_l2(out.to_nchw().cpu(), want) < ELEM_TOL[prec] * 2


@pytest.mark.parametrize("prec", list(FMTS))
@pytest.mark.parametrize("b,s,c,heads", [(2, 64, 256, 4), (3, 16, 512, 4), (2, 256, 128, 4), (1, 100, 128, 16), (2, 40, 256, 1)])
def test_attention_core(E, prec, b, s, c, heads):
    fmt = FMTS[prec]
    qkv = gen(1, 3 * c, 1, b * s, seed=1)
    if prec != "fp32":
        qkv = act_of(E, qkv, fmt).to_nchw().cpu()
    tok = qkv[0, :, 0].T.reshape(b, s, 3 * c)
    d = c // heads
    q, k, v = (z.reshape(b, s, heads, d).permute(0, 2, 1, 3) for z in tok.chunk(3, dim=-1))
    want = (torch.softmax(q @ k.transpose(-1, -2) / math.sqrt(d), -1) @ v).permute(0, 2, 1, 3).reshape(b * s, c)
    out = E.Kernels(fmt, torch.device("cuda")).attention_core(act_of(E, qkv, fmt), b, s, c, heads)
    got = out.to_nchw().cpu()[0, :, 0].T
    assert rel_l2(got, want) < {"fp32": 1e-5, "bf16x3": 3e-5, "bf16": 8e-3, "fp16x2": 5e-4}[prec]


@pytest.mark.parametrize("prec", list(FMTS))
def test_final_conv(E, prec):
    from sbgm_danra_b200._lib import call
    fmt = FMTS[prec]
    n, h = 3, 32
    x = gen(n, 64, h, h, seed=1)
    if prec != "fp32":
        x = act_of(E, x, fmt).to_nchw().cpu()
    w, bias, inv = gen(1, 64, 3, 3, seed=2, scale=0.05), gen(1, seed=3), torch.tensor([0.5, 2.0, 10.0])
    want = F.conv2d(x, w, bias, padding=1) * inv[:, None, None, None]
    a = act_of(E, x, fmt)
    wp = w.permute(0, 2, 3, 1).reshape(1, 9, 64).contiguous().cuda()
    out = torch.empty(n, 1, h, h, device="cuda")
    bias_d, inv_d = bias.cuda(), inv.cuda()      # keep the device copies alive across the launch
    call("sbgm_final_conv", a.ptr, a.plane, fmt, wp.data_ptr(), bias_d.data_ptr(), inv_d.data_ptr(), 1, 0, None,
         out.data_ptr(), n, h, h, 64, 1, torch.cuda.current_stream().cuda_stream)
    assert rel_l2(out.cpu(), want) < 1e-5


def test_philox_matches_numpy_restatement():
    from oracle import philox_ref
    from sbgm_danra_b200._lib import call
    st = torch.cuda.current_stream().cuda_stream
    for count, first in ((4096, 0), (1001, 64)):
        out = torch.empty(count, device="cuda")
        call("sbgm_philox_normal", out.data_ptr(), count, 0x1234567890ABCDEF, 5, first, st)
        want = philox_ref.normal(count, 0x1234567890ABCDEF, 5, first)
        np.testing.assert_allclose(out.cpu().numpy(), want, rtol=0, atol=3e-6)
        call("sbgm_philox_uniform", out.data_ptr(), count, 99, 2, first, st)
        np.testing.assert_array_equal(out.cpu().numpy(), philox_ref.uniform(count, 99, 2, first))   # bit-exact


def test_sampler_update_kernels():
    from oracle import philox_ref
    from sbgm_danra_b200._lib import STEP_COLS, call
    st = torch.cuda.current_stream().cuda_stream
    b, per, seed = 3, 32 * 32, 77
    x0, s = gen(b, 1, 32, 32, seed=1), gen(b, 1, 32, 32, seed=2)
    s_d = s.cuda()
    table = torch.zeros(4, STEP_COLS)
    table[:, 4] = torch.tensor([0.3, 0.2, 0.1, 0.05])
    table[:, 5] = torch.tensor([0.9, 0.7, 0.5, 0.3])
    tab, counter = table.cuda(), torch.tensor([2, 0, seed, 0], dtype=torch.int32, device="cuda")
    x, mean = x0.cuda().clone(), torch.empty(b, 1, 32, 32, device="cuda")
    first = 5 * per   # this shard starts at global member 5
    call("sbgm_sampler_predictor", x.data_ptr(), s_d.data_ptr(), mean.data_ptr(), x.numel(), tab.data_ptr(),
         counter.data_ptr(), 1, 1, first, st)
    z = torch.from_numpy(philox_ref.normal(b * per, seed, 1 + 2, first)).reshape(x0.shape)
    want_mean = x0 + 0.1 * s
    assert rel_l2(mean.cpu(), want_mean) < 1e-6
    assert rel_l2(x.cpu(), want_mean + 0.5 * z) < 1e-6
    assert counter.cpu().tolist() == [3, 0, seed, 0]
    # corrector
    sumsq = torch.empty(b, device="cuda")
    call("sbgm_sampler_sumsq", s_d.data_ptr(), sumsq.data_ptr(), b, per, st)
    np.testing.assert_allclose(sumsq.cpu().numpy(), (s.reshape(b, -1) ** 2).sum(1).numpy(), rtol=1e-5)
    x = x0.cuda().clone()
    call("sbgm_sampler_corrector", x.data_ptr(), s_d.data_ptr(), sumsq.data_ptr(), b, per, 0.16, x.numel(),
         counter.data_ptr(), 1, 2, first, st)
    gn = torch.norm(s.reshape(b, -1), dim=-1).mean()
    eps = 2 * (0.16 * math.sqrt(per) / gn) ** 2
    z = torch.from_numpy(philox_ref.normal(b * per, seed, 1 + 2 * 3, first)).reshape(x0.shape)
    assert rel_l2(x.cpu(), x0 + eps * s + torch.sqrt(2 * eps) * z) < 1e-6


def test_dsm_kernels():
    from oracle import philox_ref
    from sbgm_danra_b200 import _lib
    from sbgm_danra_b200._lib import call
    st = torch.cuda.current_stream().cuda_stream
    n, per, seed = 4, 32 * 32, 11
    x, std = gen(n, 1, 32, 32, seed=1), torch.tensor([0.1, 1.0, 5.0, 20.0])
    xt, z = torch.empty(n, 1, 32, 32, device="cuda"), torch.empty(n, 1, 32, 32, device="cuda")
    x_d, std_d = x.cuda(), std.cuda()
    call("sbgm_dsm_perturb", x_d.data_ptr(), std_d.data_ptr(), xt.data_ptr(), z.data_ptr(), n, per, seed, 1, 0, st)
    zr = torch.from_numpy(philox_ref.normal(n * per, seed, 1)).reshape(x.shape)
    assert rel_l2(z.cpu(), zr) < 1e-6 and rel_l2(xt.cpu(), x + std[:, None, None, None] * zr) < 1e-6
    score, sdf = gen(n, 1, 32, 32, seed=3), gen(n, 1, 32, 32, seed=4)
    partials = torch.empty(_lib.query("sbgm_dsm_scratch_floats", n * per), device="cuda")
    loss = torch.empty((), device="cuda")
    score_d, sdf_d = score.cuda(), sdf.cuda()
    for sd_ in (sdf, None):
        call("sbgm_dsm_loss", score_d.data_ptr(), std_d.data_ptr(), z.data_ptr(),
             None if sd_ is None else sdf_d.data_ptr(), n, per, partials.data_ptr(), loss.data_ptr(), st)
        w = torch.sigmoid(sd_) * 0.5 + 0.5 if sd_ is not None else torch.ones_like(x)
        want = torch.mean(torch.sum(w * (score * std[:, None, None, None] + zr) ** 2, dim=(1, 2, 3)))
        assert abs(loss.item() - want.item()) / want.item() < 1e-5


@pytest.mark.parametrize("prec", ["bf16", "bf16x3", "fp16x2"])
@pytest.mark.parametrize("kernel", ["c64", "generic"])
def test_projection_epilogue_and_gather(E, prec, kernel):
    """conv_up (64->64) with the projection epilogue + sbgm_final_gather == conv3x3(64->1)(conv3x3(64->64)(x))."""
    from sbgm_danra_b200._lib import call
    fmt = FMTS[prec]
    n, h, w = (3, 16, 32) if kernel == "c64" else (3, 12, 20)     # 12x20 is not tileable by 8x16 -> generic kernel
    x = gen(n, 64, h, w, seed=1)
    w1, b1 = gen(64, 64, 3, 3, seed=2, scale=0.05), gen(64, seed=3, scale=0.1)
    w2, b2 = gen(1, 64, 3, 3, seed=4, scale=0.05), gen(1, seed=5)
    inv = torch.tensor([0.5, 2.0, 10.0])
    want = F.conv2d(F.conv2d(x, w1, b1, padding=1), w2, b2, padding=1) * inv[:, None, None, None]
    kern = E.Kernels(fmt, torch.device("cuda"))
    cw = E._Packer({"w": w1, "b": b1}, fmt, torch.device("cuda")).conv("w", "b")
    pw = w2.permute(0, 2, 3, 1).reshape(9, 64).contiguous().cuda()
    pr = kern.conv(act_of(E, x, fmt), cw, pad=1, proj=pw)
    b2_d, inv_d = b2.cuda(), inv.cuda()
    out = torch.empty(n, 1, h, w, device="cuda")
    call("sbgm_final_gather", pr.data_ptr(), b2_d.data_ptr(), inv_d.data_ptr(), 1, 0, None, out.data_ptr(), n, h, w,
         torch.cuda.current_stream().cuda_stream)
    assert rel_l2(out.cpu(), want) < TOL[prec]


@pytest.mark.parametrize("prec", ["bf16", "bf16x3", "fp16x2"])
@pytest.mark.parametrize("shape", [(3, 32, 32, 64, 64, True), (40, 16, 16, 128, 128, True), (160, 8, 8, 256, 512, True),
                                   (3, 16, 16, 128, 128, False),    # small grid -> split-K -> statistics not fused
                                   (2, 12, 24, 64, 128, False)],    # tile spans several partial images
                         ids=lambda t: "x".join(map(str, t)))
def test_conv_fused_groupnorm_statistics(E, prec, shape):
    """GroupNorm from the statistics emitted by a conv epilogue == GroupNorm of that conv's output
    (persistent 64->64 kernel; generic kernel with one image per tile and with several images per tile)."""
    fmt = FMTS[prec]
    n, h, w, cin, cout, fused = shape
    x = gen(n, cin, h, w, seed=1)
    w1, b1 = gen(cout, cin, 3, 3, seed=2, scale=1.0 / math.sqrt(9 * cin)), gen(cout, seed=3, scale=0.5)
    gamma, beta = 1 + 0.2 * gen(cout, seed=4), gen(cout, seed=5, scale=0.2)
    kern = E.Kernels(fmt, torch.device("cuda"))
    cw = E._Packer({"w": w1, "b": b1}, fmt, torch.device("cuda")).conv("w", "b")
    y, stats = kern.conv(act_of(E, x, fmt), cw, pad=1, gn_stats=True)
    assert (stats is not None) == fused
    got = kern.groupnorm(y, gamma.cuda(), beta.cuda(), 8, stats=stats).to_nchw().cpu()
    want = F.group_norm(y.to_nchw().cpu(), 8, gamma, beta, 1e-5)
    assert rel_l2(got, want) < {"bf16": 8e-3, "bf16x3": 3e-5, "fp16x2": 5e-4}[prec]


# ---- entry points added for the training step / tensor-core stem -------------------------------------------------
@pytest.mark.parametrize("prec", ["bf16x3", "bf16"])
def test_pack_weights_batched_matches_torch(prec):
    """sbgm_pack_weights (one launch, job table as kernel parameter) and sbgm_pack_weight against a torch restatement:
    forward orientation, transposed / tap-sliced orientation (the data-gradient weights)."""
    from sbgm_danra_b200 import train_engine as T
    fmt = FMTS[prec]
    plan = T.PackPlan(fmt)
    cases = [(gen(64, 128, 3, 3, seed=1).cuda(), list(range(9)), False), (gen(128, 64, 3, 3, seed=2).cuda(), [8, 6, 2, 0], True),
             (gen(256, 64, 1, 1, seed=3).cuda(), [0], True), (gen(64, 64, 8, 8, seed=4).cuda(), list(range(64)), False)]
    outs = [plan.add(w, taps, tr) for w, taps, tr in cases]
    plan.run()
    for (w, taps, tr), out in zip(cases, outs):
        cout, cin = w.shape[:2]
        sel = w.reshape(cout, cin, -1)[:, :, taps]                                  # [co][ci][t]
        want = (sel.permute(1, 2, 0) if tr else sel.permute(0, 2, 1)).reshape(cin if tr else cout, -1)
        single = T._pack_tc(w, fmt, taps, tr)
        assert torch.equal(out, single)
        got = (out[0].float() + out[1].float()) if fmt == 2 else out.float()
        assert rel_l2(got.cpu(), want.cpu()) < ELEM_TOL[prec]


@pytest.mark.parametrize("prec", ["bf16x3", "bf16", "fp16x2"])
@pytest.mark.parametrize("cc,bcast,size", [(1, True, 64), (6, False, 32), (0, False, 96)])
def test_stem_im2col_matches_unfold(E, prec, cc, bcast, size):
    fmt = FMTS[prec]
    n = 3
    x = gen(n, 1, size, size, seed=1)
    planes = gen(1 if bcast else n, cc, size, size, seed=2) if cc else None
    k = E.Kernels(fmt, torch.device("cuda"))
    col = k.stem_im2col(x.cuda(), None if planes is None else planes.cuda(), 0, cc + 1, cc).to_nchw().cpu()
    full = x if planes is None else torch.cat([x, planes.expand(n, -1, -1, -1)], 1)
    want = F.unfold(full, kernel_size=8, padding=3, stride=2).reshape(n, (cc + 1) * 64, size // 2, size // 2)
    assert rel_l2(col, want) < ELEM_TOL[prec]


@pytest.mark.parametrize("prec", ["bf16x3", "bf16", "fp16x2"])
def test_conv2d_tc_ex_scatter_is_conv_transpose(E, prec):
    """Four scattered 1x1 convolutions (out_step 2, offsets (a, b)) = ConvTranspose2d(kernel 2, stride 2) with bias."""
    from sbgm_danra_b200._lib import call
    fmt = FMTS[prec]
    n, c_in, c_out, h, w = 2, 128, 64, 6, 10
    x, wt, bias = gen(n, c_in, h, w, seed=1), gen(c_in, c_out, 2, 2, seed=2, scale=c_in ** -0.5), gen(c_out, seed=3, scale=0.1)
    xa = act_of(E, x, fmt)
    out = E.Act(fmt, n, 2 * h, 2 * w, c_out, torch.device("cuda"))
    bd = bias.cuda()
    for a in range(2):
        for b in range(2):
            km = wt[:, :, a, b].t().contiguous().cuda()
            packed = E.pack_tc_matrix(km, fmt)
            call("sbgm_conv2d_tc_ex", xa.ptr, xa.plane, packed.data_ptr(), c_out * c_in, bd.data_ptr(), None, 0, 0, None, 0, out.ptr, out.plane,
                 fmt, n, h, w, c_in, c_out, 1, 1, 1, 0, 0, h, w, 2 * h, 2 * w, 2, a, b, 0, None, 0, torch.cuda.current_stream().cuda_stream)
    want = F.conv_transpose2d(xa.to_nchw().cpu(), wt, bias, stride=2)
    assert rel_l2(out.to_nchw().cpu(), want) < TOL[prec]


def test_fp16x2_weight_lo_plane_carries_the_residual(E):
    """The float16 weight planes are hi | lo * 2^11.  With weights so small that the hi plane is subnormal float16 (spacing
    2^-24, i.e. ~1e-3 relative here) the product must still be exact to output rounding: the lo plane carries the residual.
    Activations are chosen exactly representable so that the only other rounding is the float16 store of the result.
    Also checks the saturating store: results beyond the float16 range clamp to +-65504 instead of becoming inf."""
    n, c, h = 2, 64, 16
    x = torch.round(gen(n, c, h, h, seed=1) * 2.0) * 32.0
    tiny = gen(64, c, 1, 1, seed=2) * 2.0 ** -16
    xa = act_of(E, x, 3)
    assert torch.equal(xa.to_nchw().cpu(), x)
    k = E.Kernels(3, torch.device("cuda"))
    want = F.conv2d(x.double(), tiny.double())
    hi_only = F.conv2d(x.double(), tiny.half().double())
    assert rel_l2(hi_only, want) > 6e-4                                        # the case discriminates
    got = k.conv(xa, E._Packer({"w": tiny}, 3, torch.device("cuda")).conv("w")).to_nchw().cpu().double()
    err = rel_l2(got, want)
    print(f"fp16x2 subnormal-hi weights: rel-L2 {err:.2e} (hi plane alone: {rel_l2(hi_only, want):.2e})")
    assert err < 3e-4
    big = k.conv(act_of(E, gen(n, c, h, h, seed=3), 3), E._Packer({"w": gen(64, c, 1, 1, seed=4) * 4096.0}, 3, torch.device("cuda")).conv("w"))
    big = big.to_nchw().cpu()
    assert torch.isfinite(big).all() and float(big.abs().max()) == 65504.0


@pytest.mark.parametrize("prec", ["fp16x2", "bf16"])
@pytest.mark.parametrize("b,s,c,heads", [(2, 64, 256, 4), (4, 64, 256, 4), (3, 64, 256, 4), (8, 16, 128, 4), (5, 16, 256, 8), (2, 256, 128, 4),
                                         (1, 256, 256, 4), (1, 128, 128, 2), (3, 32, 128, 4), (64, 4, 128, 4)])
def test_attention_out_proj_fused_kernel(E, prec, b, s, c, heads):
    """csrc/attn_fused.cu: x + out_proj(softmax(Q K^T / sqrt(d)) V) in one tcgen05 kernel (scores / probabilities in TMEM and
    shared memory) against torch fp32 on the stored operands, and against the two-launch path it replaces.  Shapes: two images
    per query tile, partial last tile (3 x 64 tokens), 8 and 32 images per tile, 16 x 16 maps (two query tiles per image),
    one image per tile, head dims 32 and 64."""
    fmt = FMTS[prec]
    dev = torch.device("cuda")
    k = E.Kernels(fmt, dev)
    from sbgm_danra_b200 import _lib
    assert _lib.query("sbgm_attention_out_proj_supported", fmt, b, s, c, heads)
    qkv = gen(1, 3 * c, 1, b * s, seed=1)
    x = gen(1, c, 1, b * s, seed=2)
    w, bias = gen(c, c, seed=3, scale=c ** -0.5), gen(c, seed=4, scale=0.1)
    qa, xa = act_of(E, qkv, fmt), act_of(E, x, fmt)
    qs, xs = qa.to_nchw().cpu()[0, :, 0].T, xa.to_nchw().cpu()[0, :, 0].T            # what the kernel reads
    d = c // heads
    q, kk, v = (z.reshape(b, s, heads, d).permute(0, 2, 1, 3) for z in qs.reshape(b, s, 3 * c).chunk(3, dim=-1))
    att = (torch.softmax(q @ kk.transpose(-1, -2) / math.sqrt(d), -1) @ v).permute(0, 2, 1, 3).reshape(b * s, c)
    want = xs + att @ w.T + bias
    cw = E._Packer({"w": w, "b": bias}, fmt, dev).conv("w", "b")
    got = k.attention_out_proj(qa, xa, cw, b, s, c, heads).to_nchw().cpu()[0, :, 0].T
    err = rel_l2(got, want)
    two = k.linear(k.attention_core(qa, b, s, c, heads), cw, residual=xa).to_nchw().cpu()[0, :, 0].T
    print(f"attention + out-proj fused [{prec}] b={b} s={s} c={c} heads={heads}: rel-L2 {err:.2e} (two-launch path {rel_l2(two, want):.2e})")
    assert err < {"fp16x2": 8e-4, "bf16": 8e-3}[prec]


@pytest.mark.parametrize("prec", ["fp16x2", "bf16x3", "bf16"])
@pytest.mark.parametrize("rows,cin,cout,act", [(4096, 256, 768, 0), (200, 128, 128, 3), (1024, 512, 1536, 0), (16384, 128, 384, 0),
                                               (77, 256, 256, 3)])
def test_linear_with_folded_layernorm(E, prec, rows, cin, cout, act):
    """sbgm_linear_ln_tc: act(LayerNorm(x) W^T + b) with the LayerNorm folded into the GEMM (per-token statistics computed in the
    kernel from the operand tiles, y = rstd (x W'^T - mean colsum) + b') against torch on the stored input, and against the
    LayerNorm kernel + Linear pair it replaces.  x carries a per-token offset so that the cancellation mean * colsum matters."""
    fmt = FMTS[prec]
    dev = torch.device("cuda")
    x = gen(1, cin, 1, rows, seed=1) * 1.5 + gen(1, 1, 1, rows, seed=5) * 2.0 + 0.7
    w, b = gen(cout, cin, seed=2, scale=cin ** -0.5), gen(cout, seed=3, scale=0.1)
    g, beta = 1 + 0.2 * gen(cin, seed=4), gen(cin, seed=6, scale=0.2)
    xa = act_of(E, x, fmt)
    xs = xa.to_nchw().cpu()[0, :, 0].T
    want = F.linear(F.layer_norm(xs, (cin,), g, beta, 1e-5), w, b)
    want = F.gelu(want) if act == 3 else want
    pk = E._Packer({"w": w, "b": b, "g": g, "beta": beta}, fmt, dev)
    k = E.Kernels(fmt, dev)
    got = k.linear_ln(xa, E.pack_linear_ln(pk, "w", "b", "g", "beta"), act=act).to_nchw().cpu()[0, :, 0].T
    two = k.linear(k.layernorm(xa, g.cuda(), beta.cuda()), pk.conv("w", "b"), act=act).to_nchw().cpu()[0, :, 0].T
    err, err2 = rel_l2(got, want), rel_l2(two, want)
    print(f"LayerNorm-folded Linear [{prec}] {rows}x{cin}->{cout} act={act}: rel-L2 {err:.2e} (LayerNorm kernel + Linear: {err2:.2e})")
    assert err < {"fp16x2": 6e-4, "bf16x3": 1e-4, "bf16": 2e-2}[prec] and err < 2.0 * err2 + 1e-5


@pytest.mark.parametrize("prec", ["fp16x2", "bf16x3", "bf16"])
@pytest.mark.parametrize("n,size,bcast,with_partial", [(3, 64, True, True), (2, 32, False, True), (5, 96, True, True), (2, 128, True, False),
                                                       (70, 32, True, True)])
def test_stem_fused_window_kernel(E, prec, n, size, bcast, with_partial):
    """sbgm_stem_x_tc: conv1 on the noisy-field channel with the 8x8 stride-2 windows built in shared memory (no im2col tensor),
    + the conditioning partial sums (broadcast or per member) + the time projection, against F.conv2d; also against the
    im2col + 1x1 path it replaces."""
    from sbgm_danra_b200._lib import call
    fmt = FMTS[prec]
    dev = torch.device("cuda")
    x = gen(n, 1, size, size, seed=1) * 9.0
    w = gen(64, 1, 8, 8, seed=2, scale=0.1)
    partial = gen(1 if bcast else n, 64, size // 2, size // 2, seed=3) if with_partial else None
    tproj = gen(n, 80, seed=4)
    pa = None if partial is None else act_of(E, partial, fmt)
    ps = 0.0 if partial is None else pa.to_nchw().cpu()
    want = F.conv2d(x, w, stride=2, padding=3) + ps + tproj[:, 8:72, None, None]
    cw = E.ConvW(E.pack_tc_matrix(w.reshape(64, 64).contiguous().cuda(), fmt), None, 64, 64, 1, 1)
    out = E.Act(fmt, n, size // 2, size // 2, 64, dev)
    xd, td = x.cuda(), tproj.cuda()
    tv = td[:, 8:72]
    call("sbgm_stem_x_tc", xd.data_ptr(), cw.w.data_ptr(), cw.plane, None if pa is None else pa.ptr, 0 if pa is None else pa.plane,
         0 if pa is None else pa.n, tv.data_ptr(), tv.stride(0), out.ptr, out.plane, fmt, n, size, size, torch.cuda.current_stream().cuda_stream)
    err = rel_l2(out.to_nchw().cpu(), want)
    print(f"fused stem [{prec}] n={n} {size}x{size}: rel-L2 {err:.2e}")
    assert err < TOL[prec]


@pytest.mark.parametrize("prec", ["fp16x2", "bf16"])
@pytest.mark.parametrize("case", [
    (64, 32, 32, 128, 128, 3, 1, 1, "full"),      # slab mode, 512 tiles: two tiles per CTA at 128 wide
    (64, 32, 32, 128, 64, 3, 1, 1, "plain"),      # 64-wide
    (64, 16, 16, 256, 256, 3, 1, 1, "relu"),      # 256 CTAs
    (64, 8, 8, 512, 512, 3, 1, 1, "plain"),       # 8 x 8 maps (tiles of two images): 128 CTAs -> 64-wide tiles, two per CTA
    (33, 8, 8, 256, 256, 3, 1, 1, "full"),        # odd image count: the last CTA's second tile lies outside the tensor
    (64, 64, 64, 64, 64, 8, 2, 3, "relu"),        # plain mode, strided (Encoder.conv2)
    (7, 32, 32, 128, 128, 3, 1, 1, "gelu"),       # odd tile count in slab mode
    (64, 16, 16, 128, 256, 3, 2, 1, "relu"),      # strided 3 x 3
], ids=lambda c: "x".join(map(str, c)))
def test_conv2d_two_pixel_tiles_per_cta(E, prec, case, monkeypatch):
    """The MT = 2 kernels (two 128-pixel tiles per CTA sharing every weight box) against torch, with the fused GroupNorm statistics
    where the layer has them.  The cases are shapes that the grid-size rule (>= 252 one-tile CTAs) sends to MT = 2."""
    n, h, w, cin, cout, k, stride, pad, epi = case
    fmt = FMTS[prec]
    x = gen(n, cin, h, w, seed=1)
    wt = gen(cout, cin, k, k, seed=2, scale=1.0 / math.sqrt(cin * k * k))
    bias = gen(cout, seed=3, scale=0.1) if epi != "plain" else None
    ho, wo = (h + 2 * pad - k) // stride + 1, (w + 2 * pad - k) // stride + 1
    res = gen(n, cout, ho, wo, seed=4) if epi == "full" else None
    tproj = gen(n, cout + 16, seed=5) if epi == "full" else None
    act = {"plain": 0, "full": 1, "relu": 1, "gelu": 3}[epi]
    want = F.conv2d(x, wt, bias, stride=stride, padding=pad)
    if res is not None:
        want = want + res
    want = {0: lambda v: v, 1: F.relu, 3: F.gelu}[act](want)
    if tproj is not None:
        want = want + tproj[:, 8:8 + cout, None, None]
    kern = E.Kernels(fmt, torch.device("cuda"))
    sd = {"w": wt}
    if bias is not None:
        sd["b"] = bias
    cw = E._Packer(sd, fmt, torch.device("cuda")).conv("w", "b" if bias is not None else None)
    tp = tproj.cuda()[:, 8:8 + cout] if tproj is not None else None
    out = kern.conv(act_of(E, x, fmt), cw, stride=stride, pad=pad, act=act, residual=None if res is None else act_of(E, res, fmt), tproj=tp)
    err = rel_l2(out.to_nchw().cpu(), want)
    assert err < TOL[prec], f"rel-L2 {err:.3e}"
    if epi == "plain" and stride == 1:          # GroupNorm statistics fused into the epilogue of a two-tile CTA
        gamma, beta = 1 + 0.2 * gen(cout, seed=6), gen(cout, seed=7, scale=0.2)
        y, stats = kern.conv(act_of(E, x, fmt), cw, pad=pad, gn_stats=True)
        if stats is not None:
            got = kern.groupnorm(y, gamma.cuda(), beta.cuda(), 8, stats=stats).to_nchw().cpu()
            assert rel_l2(got, F.group_norm(y.to_nchw().cpu(), 8, gamma, beta, 1e-5)) < {"bf16": 8e-3, "fp16x2": 5e-4}[prec]


@pytest.mark.parametrize("prec", ["bf16", "fp16x2"])
@pytest.mark.parametrize("mode", ["plain", "stats", "proj"])
@pytest.mark.parametrize("shape", [(3, 8, 4), (2, 16, 16), (5, 16, 8), (150, 8, 4), (2, 24, 12)], ids=lambda t: "x".join(map(str, t)))
def test_conv_with_the_upsample_in_its_operand_stage(E, prec, mode, shape):
    """sbgm_conv3x3_c64_up == bilinear upsample -> 64 -> 64 convolution as two launches (the same fp32 interpolation expression
    and the same single rounding of the operand, so the two agree to the odd last-bit tie), and == torch on what the kernel
    reads.  Shapes: one tile per image (every halo row and column is padding or a
    clamped border tap), 2 x 4 tiles, 2 x 2, more tiles than SMs (persistent loop, stage ring and patch buffers wrap around),
    3 x 3 tiles (interior tiles on every side)."""
    fmt = FMTS[prec]
    n, hl, wl = shape
    dev = torch.device("cuda")
    kern = E.Kernels(fmt, dev)
    x = act_of(E, gen(n, 64, hl, wl, seed=1), fmt)
    w1, b1 = gen(64, 64, 3, 3, seed=4, scale=1.0 / 24), gen(64, seed=5, scale=0.1)
    cw1 = E._Packer({"w1": w1, "b1": b1}, fmt, dev).conv("w1", "b1")
    assert kern.up_fused_ok(x, cw1)
    pw = gen(9, 64, seed=10, scale=0.1).cuda() if mode == "proj" else None
    ref = kern.conv(kern.upsample2x(x), cw1, pad=1, proj=pw, gn_stats=(mode == "stats"))
    got = kern.conv_up_fused(x, cw1, proj=pw, gn_stats=(mode == "stats"))
    torch.cuda.synchronize()
    tol2 = {"bf16": 3e-4, "fp16x2": 2e-5}[prec]           # a handful of operand values that round the other way
    want = F.conv2d(F.interpolate(x.to_nchw().cpu(), scale_factor=2, mode="bilinear", align_corners=False), w1, b1, padding=1)
    if mode == "proj":
        assert rel_l2(got[..., :9].cpu(), ref[..., :9].cpu()) < tol2
        wp = torch.einsum("nchw,qc->nhwq", want, pw.cpu())
        assert rel_l2(got[..., :9].cpu(), wp) < {"bf16": 1.2e-2, "fp16x2": 1e-3}[prec]
    else:
        a, b = (got[0], ref[0]) if mode == "stats" else (got, ref)
        assert rel_l2(a.to_nchw().cpu(), b.to_nchw().cpu()) < tol2
        assert rel_l2(a.to_nchw().cpu(), want) < {"bf16": 1.2e-2, "fp16x2": 1e-3}[prec]
        if mode == "stats":      # the statistics describe the tensor this kernel stored
            gamma, beta = 1 + 0.2 * gen(64, seed=6), gen(64, seed=7, scale=0.2)
            y = kern.groupnorm(a, gamma.cuda(), beta.cuda(), 8, stats=got[1]).to_nchw().cpu()
            assert rel_l2(y, F.group_norm(a.to_nchw().cpu(), 8, gamma, beta, 1e-5)) < {"bf16": 8e-3, "fp16x2": 5e-4}[prec]
