"""CPU: the parity-class decomposition behind the stem's data-gradient kernels (sbgm_stem_dgrad_tc / _simt), restated in torch.

Encoder.conv1 is 8x8, stride 2, pad 3.  Input pixel (2 j + py, 2 i + px) receives df[j + py - 2 + ky][i + px - 2 + kx] times the
weight tap train_engine.stem_dgrad_taps(py, px)[ky * 4 + kx]; summed over the 16 taps and the 64 channels this must be
torch.nn.grad.conv2d_input in float64."""
import pytest
import torch


def _class_dgrad(df, w, py, px):
    from sbgm_danra_b200.train_engine import stem_dgrad_taps
    n, _, hh, wh = df.shape
    cin = w.shape[1]
    taps = stem_dgrad_taps(py, px)
    pad = torch.nn.functional.pad(df, (2, 2, 2, 2))           # offsets -2..2 around each class position
    out = torch.zeros(n, cin, hh, wh, dtype=df.dtype)
    for t, tap in enumerate(taps):
        ky, kx = divmod(t, 4)
        oy, ox = py - 2 + ky, px - 2 + kx
        win = pad[:, :, 2 + oy:2 + oy + hh, 2 + ox:2 + ox + wh]
        out += torch.einsum("nchw,ci->nihw", win, w[:, :, tap // 8, tap % 8])
    return out


@pytest.mark.parametrize("cin,size", [(1, 16), (7, 32), (15, 24)])
def test_parity_classes_rebuild_conv2d_input(cin, size):
    g = torch.Generator().manual_seed(cin)
    n = 2
    w = torch.randn(64, cin, 8, 8, generator=g, dtype=torch.float64)
    df = torch.randn(n, 64, size // 2, size // 2, generator=g, dtype=torch.float64)
    ref = torch.nn.grad.conv2d_input((n, cin, size, size), w, df, stride=2, padding=3)
    got = torch.empty_like(ref)
    for py in range(2):
        for px in range(2):
            got[:, :, py::2, px::2] = _class_dgrad(df, w, py, px)
    assert torch.allclose(got, ref, rtol=0, atol=1e-10)


def test_taps_are_the_kernels_order():
    from sbgm_danra_b200.train_engine import stem_dgrad_taps
    # r = 7 - py - 2 ky, s = 7 - px - 2 kx (include/sbgm_b200.h, sbgm_stem_dgrad_tc)
    for py in range(2):
        for px in range(2):
            assert stem_dgrad_taps(py, px) == [(7 - py - 2 * ky) * 8 + 7 - px - 2 * kx for ky in range(4) for kx in range(4)]
