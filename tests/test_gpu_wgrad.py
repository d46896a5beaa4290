"""GPU: the weight-gradient kernels against a float64 reference, at every tensor-core weight-gradient shape of the benchmarked
C4 training step and at the edges of the kernels' tilings.

Three kernels compute dW[co][ci][r][s] = sum over output pixels p of dy[p][co] * x[p * stride + (r, s) - pad][ci]:
  slab      conv_wgrad_tc.cu's conv_wgrad_slab_kernel: bf16 3x3 stride-1 layers whose CTAs get >= 8 16x8-pixel tiles each
  unit64    conv_wgrad_tc_kernel with 64 output channels per CTA (bf16 with cout % 128 != 0, and every bf16x3 layer)
  unit128   conv_wgrad_tc_kernel with 128 output channels per CTA (bf16, cout % 128 == 0)
  SIMT      conv_grad_simt.cu's CUDA-core kernel (the fp32 path and the cross-check)
Each case names the route it exists for in bf16 (bf16x3 always takes unit64) and asserts it through sbgm_conv2d_wgrad_tc_plan
before it compares anything, so a change of the dispatch rule cannot quietly move a case off the kernel it was written for.

The reference is torch.nn.grad.conv2d_weight in float64 on the values the kernels read (the activation format's stored
operands).  A bf16 x bf16 product is exact in fp32, so the only error left is fp32 summation, and the gates are tight:
  bf16 (tensor cores)  1e-5
  bf16x3               5e-5   the lo x lo product is dropped: about 2^-16 of each product
  SIMT                 1e-5   fp32 FMA over the same operands
Every case also shows that its gate can fail: leaving out the last pixel split's tiles changes the reference by more than 10x
the gate.  The workspace and dW start as NaN, so a partial sum that is never written fails the finiteness check, and two calls
must agree bit for bit (multi-GPU parity and CUDA-graph replay rely on the fixed-order split reduction).
"""
import ctypes

import pytest
import torch

from conftest import rel_l2

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
FMTS = {"bf16": 1, "bf16x3": 2}
GATE = {"bf16": 1e-5, "bf16x3": 5e-5}
SIMT_GATE = 1e-5
ROUTES = {(1, 64): "slab", (0, 64): "unit64", (0, 128): "unit128"}        # (kernel, output channels per CTA) of the plan

# Every tensor-core weight gradient of the C4 training step (bench.py's train_c4: 128x128 fields, Cin = 7 + seasons, bf16,
# batch 64), each shape once: (n, h, w, cin, cout, k, stride, pad) of the layer input x, and the bf16 route.
# test_table_lists_every_tensor_core_wgrad_of_the_c4_step checks this table against the calls one step makes.
C4 = {
    "stem_im2col_64x64": ((64, 64, 64, 448, 64, 1, 1, 0), "unit64"),      # Encoder.conv1 as a 1x1 over the im2col tensor
    "enc_conv2_8x8s2": ((64, 64, 64, 64, 64, 8, 2, 3), "unit64"),
    "enc_layer1_32x32": ((64, 32, 32, 64, 64, 3, 1, 1), "unit64"),
    "enc_layer2_conv1_s2": ((64, 32, 32, 64, 128, 3, 2, 1), "unit128"),
    "enc_layer2_down_1x1s2": ((64, 32, 32, 64, 128, 1, 2, 0), "unit128"),
    "enc_layer2_16x16": ((64, 16, 16, 128, 128, 3, 1, 1), "unit128"),
    "enc_layer3_conv1_s2": ((64, 16, 16, 128, 256, 3, 2, 1), "unit128"),
    "enc_layer3_down_1x1s2": ((64, 16, 16, 128, 256, 1, 2, 0), "unit128"),
    "enc_layer3_8x8": ((64, 8, 8, 256, 256, 3, 1, 1), "unit128"),
    "enc_layer4_conv1_s2": ((64, 8, 8, 256, 512, 3, 2, 1), "unit128"),
    "enc_layer4_down_1x1s2": ((64, 8, 8, 256, 512, 1, 2, 0), "unit128"),
    "enc_layer4_4x4": ((64, 4, 4, 512, 512, 3, 1, 1), "unit128"),
    "attn256_in_proj": ((1, 1, 4096, 256, 768, 1, 1, 0), "unit128"),      # attention at 8x8: 4096 tokens (encoder 3, decoder 0)
    "attn256_proj": ((1, 1, 4096, 256, 256, 1, 1, 0), "unit128"),         # out_proj, ff.0, ff.2
    "attn512_in_proj": ((1, 1, 1024, 512, 1536, 1, 1, 0), "unit128"),     # attention at 4x4 (encoder 4)
    "attn512_proj": ((1, 1, 1024, 512, 512, 1, 1, 0), "unit128"),
    "attn128_in_proj": ((1, 1, 16384, 128, 384, 1, 1, 0), "unit128"),     # attention at 16x16 (decoder 1)
    "attn128_proj": ((1, 1, 16384, 128, 128, 1, 1, 0), "unit128"),
    # a decoder block: conv_up keeps the input's channels (after the 2x upsample), conv maps them to the block's output
    "dec0_conv_up_8x8": ((64, 8, 8, 512, 512, 3, 1, 1), "unit128"),
    "dec0_conv_8x8": ((64, 8, 8, 512, 256, 3, 1, 1), "unit128"),
    "dec1_conv_up_16x16": ((64, 16, 16, 256, 256, 3, 1, 1), "slab"),
    "dec1_conv_16x16": ((64, 16, 16, 256, 128, 3, 1, 1), "unit128"),
    "dec2_conv_up_32x32": ((64, 32, 32, 128, 128, 3, 1, 1), "slab"),
    "dec2_conv_32x32": ((64, 32, 32, 128, 64, 3, 1, 1), "unit64"),
    "dec3_64x64": ((64, 64, 64, 64, 64, 3, 1, 1), "slab"),                 # decoder block 3's conv_up and conv
    "final_conv_up_128x128": ((64, 128, 128, 64, 64, 3, 1, 1), "slab"),
}

CASES = dict(C4)
CASES.update({
    # the final layer at the per-GPU batches of the strong-scaling runs
    "final_conv_up_batch32": ((32, 128, 128, 64, 64, 3, 1, 1), "slab"),
    "final_conv_up_batch16": ((16, 128, 128, 64, 64, 3, 1, 1), "slab"),
    # slab edges
    "slab_one_tile_per_image": ((24, 16, 8, 512, 512, 3, 1, 1), "slab"),    # every halo side is padding; 8 images per split
    # 3 x 4 tiles per image, 13 tiles per split (splits start inside images), a short last split (6 tiles), 4 x 2 channel blocks
    "slab_splits_inside_images": ((20, 48, 32, 256, 128, 3, 1, 1), "slab"),
    # 2 x 6 tiles per image, 11 per split, last split 10 tiles, 2 x 3 channel blocks, odd image count
    "slab_cin_lt_cout": ((21, 32, 48, 128, 192, 3, 1, 1), "slab"),
    # per-unit edges
    "unit_odd_units_1x1": ((4, 16, 16, 64, 128, 1, 1, 0), "unit128"),      # one (tap, channel block) unit: half a CTA is padding
    "unit_odd_units_3x3": ((2, 24, 24, 64, 64, 3, 1, 1), "unit64"),        # nine units
    "unit_4x4_n3": ((3, 4, 4, 512, 512, 3, 1, 1), "unit128"),             # 4x4x8 tile holding 3 images
    "unit_8x8_n3": ((3, 8, 8, 256, 256, 3, 1, 1), "unit128"),             # 8x8x2 tiles, the second half-empty
    "unit_ragged_13x37": ((2, 13, 37, 64, 128, 3, 1, 1), "unit128"),      # 64x2 tiles: ragged columns and rows
    "unit_ragged_24x20": ((3, 24, 20, 64, 64, 3, 1, 1), "unit64"),        # 32x4 tiles over 20 columns
    "unit_ragged_s2_26x22": ((3, 26, 22, 128, 128, 3, 2, 1), "unit128"),  # stride 2 onto a 13x11 output
    # the geometries of the former tensor-core vs CUDA-core test, all on the per-unit kernel (one tile per split)
    "simt_xcheck_32x32": ((4, 32, 32, 64, 64, 3, 1, 1), "unit64"),
    "simt_xcheck_16x8": ((3, 16, 8, 128, 128, 3, 1, 1), "unit128"),
    "simt_xcheck_48x24_c192": ((5, 48, 24, 64, 192, 3, 1, 1), "unit64"),
    "simt_xcheck_c256_to_64": ((2, 32, 32, 256, 64, 3, 1, 1), "unit64"),
    "simt_xcheck_24_rows": ((2, 24, 16, 64, 64, 3, 1, 1), "unit64"),
    "simt_xcheck_s2": ((2, 16, 16, 64, 128, 3, 2, 1), "unit128"),
    # stride 2 with k = 1, 3 and 8 at small batch (the C4 table has them at batch 64)
    "unit_s2_k1": ((2, 32, 32, 64, 128, 1, 2, 0), "unit128"),
    "unit_s2_k8": ((2, 32, 32, 64, 64, 8, 2, 3), "unit64"),
})


def gen(*shape, seed=0):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed))


def out_hw(geom):
    n, h, w, cin, cout, k, stride, pad = geom
    return (h + 2 * pad - k) // stride + 1, (w + 2 * pad - k) // stride + 1


def wgrad_plan(fmt, geom):
    """sbgm_conv2d_wgrad_tc_plan: (kernel, block_n, splits, tiles_per_split, total_tiles, tile_w, tile_h, tile_n)."""
    from sbgm_danra_b200 import _lib
    n, h, w, cin, cout, k, stride, pad = geom
    plan = (ctypes.c_int * 8)()
    assert _lib.query("sbgm_conv2d_wgrad_tc_plan", fmt, n, h, w, cin, cout, k, k, stride, pad, plan) == 0, _lib.query("sbgm_last_error")
    return tuple(plan)


def last_split_mask(plan, n, ho, wo):
    """[n, 1, ho, wo]: the output pixels of the tensor-core kernel's last pixel split."""
    _, _, splits, per, total, tw_, th_, tn_ = plan
    tiles_w, tiles_h = -(-wo // tw_), -(-ho // th_)
    mask = torch.zeros(n, 1, ho, wo, dtype=torch.bool)
    for t in range((splits - 1) * per, total):
        tw, th, tn = t % tiles_w, (t // tiles_w) % tiles_h, t // (tiles_w * tiles_h)
        mask[tn * tn_:(tn + 1) * tn_, :, th * th_:(th + 1) * th_, tw * tw_:(tw + 1) * tw_] = True
    return mask


def run_wgrad(kind, fmt, xa, da, geom):
    """dW from sbgm_conv2d_wgrad_{tc,simt} with the workspace and dW filled with NaN beforehand."""
    from sbgm_danra_b200 import _lib
    from sbgm_danra_b200._lib import call
    n, h, w, cin, cout, k, stride, pad = geom
    args = (n, h, w, cin, cout, k, k, stride, pad)
    nws = _lib.query(f"sbgm_conv2d_wgrad_{kind}_workspace_floats", *(((fmt,) + args) if kind == "tc" else args))
    ws = torch.full((nws,), float("nan"), device=DEV)
    dw = torch.full((cout, cin, k, k), float("nan"), device=DEV)
    call(f"sbgm_conv2d_wgrad_{kind}", xa.ptr, xa.plane, da.ptr, da.plane, dw.data_ptr(), fmt, *args, ws.data_ptr(),
         torch.cuda.current_stream().cuda_stream)
    dw = dw.cpu()
    assert torch.isfinite(dw).all(), f"{kind}: a partial sum was never written"
    return dw


@pytest.mark.parametrize("prec", ["bf16", "bf16x3"])
@pytest.mark.parametrize("name", list(CASES))
def test_wgrad_matches_float64(prec, name):
    from sbgm_danra_b200.engine import Act
    geom, route = CASES[name]
    fmt, gate = FMTS[prec], GATE[prec]
    n, h, w, cin, cout, k, stride, pad = geom
    ho, wo = out_hw(geom)
    plan = wgrad_plan(fmt, geom)
    want_route = route if prec == "bf16" else "unit64"
    assert ROUTES.get(plan[:2]) == want_route, f"{name} [{prec}]: plan {plan} is not the {want_route} route"

    xa = Act.from_nchw(gen(n, cin, h, w, seed=1).to(DEV), fmt)
    da = Act.from_nchw(gen(n, cout, ho, wo, seed=2).to(DEV), fmt)
    x64, dy64 = xa.to_nchw().cpu().double(), da.to_nchw().cpu().double()
    ref = torch.nn.grad.conv2d_weight(x64, (cout, cin, k, k), dy64, stride=stride, padding=pad)

    # the gate can fail: dW is linear in dy, so leaving out the last split's tiles changes it by their contribution alone
    mask = last_split_mask(plan, n, ho, wo)
    first = int(mask.flatten(1).any(1).nonzero()[0])
    last_part = torch.nn.grad.conv2d_weight(x64[first:], (cout, cin, k, k), (dy64 * mask)[first:], stride=stride, padding=pad)
    dropped = rel_l2(ref - last_part, ref)
    assert dropped > 10 * gate, f"{name} [{prec}]: the last split moves dW by only {dropped:.1e}"

    tc = run_wgrad("tc", fmt, xa, da, geom)
    assert torch.equal(tc, run_wgrad("tc", fmt, xa, da, geom)), "the tensor-core weight gradient is not deterministic"
    simt = run_wgrad("simt", fmt, xa, da, geom)
    assert torch.equal(simt, run_wgrad("simt", fmt, xa, da, geom)), "the CUDA-core weight gradient is not deterministic"
    e_tc, e_simt = rel_l2(tc, ref), rel_l2(simt, ref)
    print(f"{name} {geom} [{prec}] {want_route}: splits {plan[2]} x {plan[3]} tiles of {plan[5]}x{plan[6]}x{plan[7]} "
          f"(total {plan[4]}); tc {e_tc:.2e}, simt {e_simt:.2e} (gate {gate:.0e}), last split {dropped:.1e}")
    assert e_tc < gate, f"{name} [{prec}]: tensor-core dW rel-L2 {e_tc:.2e}"
    assert e_simt < SIMT_GATE, f"{name} [{prec}]: CUDA-core dW rel-L2 {e_simt:.2e}"


def test_table_lists_every_tensor_core_wgrad_of_the_c4_step(monkeypatch):
    """C4 above is exactly the set of tensor-core weight-gradient shapes one bf16 C4 training step at batch 64 launches."""
    from oracle.synth import config_for, synth_batch, synth_state_dict
    from sbgm_danra_b200 import score_sampling, train_engine
    from sbgm_danra_b200._smoke import build_model
    from sbgm_danra_b200.score_unet import loss_fn, marginal_prob_std_fn
    seen = []
    wgrad = train_engine.TrainKernels.wgrad

    def recording(self, x, dy, dw, cin, cout, kh, kw, stride, pad):
        tc = wgrad(self, x, dy, dw, cin, cout, kh, kw, stride, pad)
        if tc:
            assert kh == kw
            seen.append((x.n, x.h, x.w, cin, cout, kh, stride, pad))
        return tc

    monkeypatch.setattr(train_engine.TrainKernels, "wgrad", recording)
    ck = dict(n_lr=2, geo=True, seasons=True)
    cfg = config_for(**ck)
    net = build_model(cfg, synth_state_dict(cfg), "bf16", DEV).train()
    b = synth_batch(batch=64, size=128, **ck)
    c = lambda v: None if v is None else v.to(DEV)
    score_sampling.manual_seed(5)
    loss_fn(net, c(b.x), marginal_prob_std_fn, y=c(b.y), cond_img=c(b.cond_img), lsm_cond=c(b.lsm_cond), topo_cond=c(b.topo_cond),
            sdf_cond=c(b.sdf_cond)).backward()
    print(f"C4 step, batch 64: {len(seen)} tensor-core weight gradients, {len(set(seen))} shapes")
    assert set(seen) == {geom for geom, _ in C4.values()}
