"""Which kernels take each conv of the models (-m "not gpu"): the dispatch queries of the library are host functions, so
this runs with or without a device.

tcgen05 takes every channel count with 16-byte NHWC rows (C % 8 == 0, C >= 16): a reduction that is not a multiple of
16 runs on 64-channel chunks (or the narrowest chunk covering it) whose last box TMA zero-fills.  The layers checked here
are derived from the models themselves (engine plans and their input maps at 128 patches), not from a hand-made list."""
import pytest

from helpers import BF16, F32, lib

import models  # noqa: E402
from svrs_native.engine import ConvOp  # noqa: E402

B = 128


def _dispatch(model):
    """[(net, kind, cin, cout, H, fprop on tcgen05, dgrad on tcgen05, wgrad packed layout)] of every conv at 128 patches."""
    eng = model._engine()
    shapes = eng.conv_input_shapes(B)
    rows = []
    for net in eng.nets.values():
        for op in net.ops:
            if not isinstance(op, ConvOp):
                continue
            n, h, w = shapes[id(op)]
            ci, co = op.cin, op.cout
            oh, ow = (h // 2, w // 2) if op.kind == "c4" else (h, w)     # conv_tc's output grid (per-parity grid for ct)
            f = lib.tc_would_run(BF16, ci, co, oh, ow)
            d = lib.tc_would_run(BF16, co, ci, oh, ow)
            if op.kind == "ct":
                wl = lib.convT2d_wgrad_layout(BF16, n, h, w, ci, co)
            else:
                wl = lib.conv2d_wgrad_layout(BF16, n, h, w, ci, co, 3 if op.kind == "c3" else 4)
            rows.append((net.name, op.kind, ci, co, h, int(f), int(d), int(wl)))
    return rows


# The parent's answers for every conv of the benchmarked models: (net, kind, cin, cout, input H, fprop, dgrad, wgrad layout)
PARENT = {
    "cond_cr2": [
        ('decoder_x', 'c3', 16, 4, 64, 1, 0, 0),
        ('decoder_x', 'c3', 16, 16, 64, 1, 1, 1),
        ('decoder_x', 'c3', 64, 16, 64, 1, 1, 1),
        ('decoder_x', 'c3', 64, 64, 64, 1, 1, 1),
        ('decoder_x', 'c3', 128, 128, 32, 1, 1, 1),
        ('decoder_x', 'c3', 256, 256, 8, 1, 1, 1),
        ('decoder_x', 'c3', 256, 256, 16, 1, 1, 1),
        ('decoder_x', 'ct', 128, 64, 32, 1, 1, 1),
        ('decoder_x', 'ct', 256, 128, 16, 1, 1, 1),
        ('decoder_x', 'ct', 256, 256, 8, 1, 1, 1),
        ('decoder_y', 'c3', 16, 4, 32, 1, 0, 0),
        ('decoder_y', 'c3', 16, 16, 32, 1, 1, 1),
        ('decoder_y', 'c3', 32, 32, 8, 1, 1, 1),
        ('decoder_y', 'c3', 64, 16, 32, 1, 1, 1),
        ('decoder_y', 'c3', 64, 64, 32, 1, 1, 1),
        ('decoder_y', 'c3', 128, 128, 16, 1, 1, 1),
        ('decoder_y', 'ct', 32, 128, 8, 1, 1, 1),
        ('decoder_y', 'ct', 128, 64, 16, 1, 1, 1),
        ('encoder_x', 'c3', 4, 4, 64, 0, 0, 0),
        ('encoder_x', 'c3', 16, 16, 32, 1, 1, 1),
        ('encoder_x', 'c3', 64, 64, 16, 1, 1, 1),
        ('encoder_x', 'c3', 128, 128, 8, 1, 1, 1),
        ('encoder_x', 'c3', 128, 256, 8, 1, 1, 1),
        ('encoder_x', 'c4', 4, 16, 64, 0, 1, 0),
        ('encoder_x', 'c4', 16, 64, 32, 1, 1, 1),
        ('encoder_x', 'c4', 64, 128, 16, 1, 1, 1),
        ('encoder_y', 'c3', 4, 4, 32, 0, 0, 0),
        ('encoder_y', 'c3', 16, 16, 16, 1, 1, 1),
        ('encoder_y', 'c3', 64, 64, 8, 1, 1, 1),
        ('encoder_y', 'c3', 64, 128, 8, 1, 1, 1),
        ('encoder_y', 'c3', 128, 64, 8, 1, 1, 1),
        ('encoder_y', 'c3', 128, 128, 8, 1, 1, 1),
        ('encoder_y', 'c4', 4, 16, 32, 0, 1, 0),
        ('encoder_y', 'c4', 16, 64, 16, 1, 1, 1),
        ('logvar_u_y_to_z', 'c3', 512, 512, 4, 1, 1, 1),
        ('logvar_u_y_to_z', 'c3', 1024, 512, 4, 1, 1, 1),
        ('mu_u_y_to_z', 'c3', 512, 512, 4, 1, 1, 1),
        ('mu_u_y_to_z', 'c3', 1024, 512, 4, 1, 1, 1),
        ('u_to_z', 'c3', 128, 128, 4, 1, 1, 1),
        ('u_to_z', 'c3', 128, 512, 4, 1, 1, 1),
        ('y_to_z', 'c3', 4, 4, 32, 0, 0, 0),
        ('y_to_z', 'c3', 16, 16, 16, 1, 1, 1),
        ('y_to_z', 'c3', 64, 64, 8, 1, 1, 1),
        ('y_to_z', 'c3', 128, 128, 4, 1, 1, 1),
        ('y_to_z', 'c3', 128, 512, 4, 1, 1, 1),
        ('y_to_z', 'c4', 4, 16, 32, 0, 1, 0),
        ('y_to_z', 'c4', 16, 64, 16, 1, 1, 1),
        ('y_to_z', 'c4', 64, 128, 8, 1, 1, 1),
    ],
    "cond_cr16": [
        ('decoder_x', 'c3', 16, 4, 64, 1, 0, 0),
        ('decoder_x', 'c3', 16, 16, 64, 1, 1, 1),
        ('decoder_x', 'c3', 32, 32, 8, 1, 1, 1),
        ('decoder_x', 'c3', 64, 16, 64, 1, 1, 1),
        ('decoder_x', 'c3', 64, 64, 64, 1, 1, 1),
        ('decoder_x', 'c3', 128, 128, 32, 1, 1, 1),
        ('decoder_x', 'c3', 256, 256, 16, 1, 1, 1),
        ('decoder_x', 'ct', 32, 256, 8, 1, 1, 1),
        ('decoder_x', 'ct', 128, 64, 32, 1, 1, 1),
        ('decoder_x', 'ct', 256, 128, 16, 1, 1, 1),
        ('decoder_y', 'c3', 4, 4, 8, 0, 0, 0),
        ('decoder_y', 'c3', 16, 4, 32, 1, 0, 0),
        ('decoder_y', 'c3', 16, 16, 32, 1, 1, 1),
        ('decoder_y', 'c3', 64, 16, 32, 1, 1, 1),
        ('decoder_y', 'c3', 64, 64, 32, 1, 1, 1),
        ('decoder_y', 'c3', 128, 128, 16, 1, 1, 1),
        ('decoder_y', 'ct', 4, 128, 8, 0, 1, 0),
        ('decoder_y', 'ct', 128, 64, 16, 1, 1, 1),
        ('encoder_x', 'c3', 4, 4, 64, 0, 0, 0),
        ('encoder_x', 'c3', 16, 16, 32, 1, 1, 1),
        ('encoder_x', 'c3', 64, 64, 16, 1, 1, 1),
        ('encoder_x', 'c3', 128, 32, 8, 1, 1, 1),
        ('encoder_x', 'c3', 128, 128, 8, 1, 1, 1),
        ('encoder_x', 'c4', 4, 16, 64, 0, 1, 0),
        ('encoder_x', 'c4', 16, 64, 32, 1, 1, 1),
        ('encoder_x', 'c4', 64, 128, 16, 1, 1, 1),
        ('encoder_y', 'c3', 4, 4, 32, 0, 0, 0),
        ('encoder_y', 'c3', 16, 16, 16, 1, 1, 1),
        ('encoder_y', 'c3', 64, 64, 8, 1, 1, 1),
        ('encoder_y', 'c3', 64, 128, 8, 1, 1, 1),
        ('encoder_y', 'c3', 128, 8, 8, 1, 0, 0),
        ('encoder_y', 'c3', 128, 128, 8, 1, 1, 1),
        ('encoder_y', 'c4', 4, 16, 32, 0, 1, 0),
        ('encoder_y', 'c4', 16, 64, 16, 1, 1, 1),
        ('logvar_u_y_to_z', 'c3', 64, 64, 4, 1, 1, 1),
        ('logvar_u_y_to_z', 'c3', 128, 64, 4, 1, 1, 1),
        ('mu_u_y_to_z', 'c3', 64, 64, 4, 1, 1, 1),
        ('mu_u_y_to_z', 'c3', 128, 64, 4, 1, 1, 1),
        ('u_to_z', 'c3', 16, 16, 4, 1, 1, 1),
        ('u_to_z', 'c3', 16, 64, 4, 1, 1, 1),
        ('y_to_z', 'c3', 4, 4, 32, 0, 0, 0),
        ('y_to_z', 'c3', 16, 16, 16, 1, 1, 1),
        ('y_to_z', 'c3', 64, 64, 8, 1, 1, 1),
        ('y_to_z', 'c3', 128, 64, 4, 1, 1, 1),
        ('y_to_z', 'c3', 128, 128, 4, 1, 1, 1),
        ('y_to_z', 'c4', 4, 16, 32, 0, 1, 0),
        ('y_to_z', 'c4', 16, 64, 16, 1, 1, 1),
        ('y_to_z', 'c4', 64, 128, 8, 1, 1, 1),
    ],
    "vae_cr2": [
        ('decoder', 'c3', 16, 4, 64, 1, 0, 0),
        ('decoder', 'c3', 16, 16, 64, 1, 1, 1),
        ('decoder', 'c3', 64, 16, 64, 1, 1, 1),
        ('decoder', 'c3', 64, 64, 64, 1, 1, 1),
        ('decoder', 'c3', 128, 128, 16, 1, 1, 1),
        ('decoder', 'c3', 128, 128, 32, 1, 1, 1),
        ('decoder', 'ct', 128, 64, 32, 1, 1, 1),
        ('decoder', 'ct', 128, 128, 16, 1, 1, 1),
        ('encoder', 'c3', 4, 4, 64, 0, 0, 0),
        ('encoder', 'c3', 16, 16, 32, 1, 1, 1),
        ('encoder', 'c3', 64, 64, 16, 1, 1, 1),
        ('encoder', 'c3', 64, 128, 16, 1, 1, 1),
        ('encoder', 'c3', 128, 128, 16, 1, 1, 1),
        ('encoder', 'c3', 128, 256, 16, 1, 1, 1),
        ('encoder', 'c4', 4, 16, 64, 0, 1, 0),
        ('encoder', 'c4', 16, 64, 32, 1, 1, 1),
    ],
}
BUILD = {"cond_cr2": lambda: models.Cond_SRVAE(2, 64), "cond_cr16": lambda: models.Cond_SRVAE(16, 64),
         "vae_cr2": lambda: models.VAE(2, 64)}


@pytest.mark.parametrize("name", sorted(PARENT))
def test_benchmarked_models_keep_their_dispatch(name):
    assert sorted(set(_dispatch(BUILD[name]()))) == sorted(PARENT[name])


# Layers that move from the CUDA-core kernels to tcgen05 (net, kind, cin, cout, input H) at the reference's own ratios.
MOVED = {
    1.5: [("encoder_x", "c3", 128, 336, 8), ("decoder_x", "c3", 336, 336, 8), ("decoder_x", "ct", 336, 256, 8),
          ("y_to_z", "c3", 128, 672, 4), ("u_to_z", "c3", 168, 168, 4), ("u_to_z", "c3", 168, 672, 4),
          ("mu_u_y_to_z", "c3", 1344, 672, 4), ("mu_u_y_to_z", "c3", 672, 672, 4),
          ("logvar_u_y_to_z", "c3", 1344, 672, 4), ("logvar_u_y_to_z", "c3", 672, 672, 4)],
    1.2: [("encoder_x", "c3", 128, 424, 8), ("decoder_x", "c3", 424, 424, 8), ("decoder_x", "ct", 424, 256, 8),
          ("y_to_z", "c3", 128, 848, 4), ("mu_u_y_to_z", "c3", 1696, 848, 4), ("mu_u_y_to_z", "c3", 848, 848, 4),
          ("logvar_u_y_to_z", "c3", 1696, 848, 4), ("logvar_u_y_to_z", "c3", 848, 848, 4)],
}


@pytest.mark.parametrize("cr", [1.5, 1.2])
def test_reference_ratios_run_on_tcgen05(cr):
    """At cr 1.5 / 1.2 every conv whose channel counts are multiples of 8 (and not the 4-channel image layers, which the
    narrow kernels take) runs fprop, dgrad and wgrad on tcgen05; the layers with 42 / 84 / 53 / 106 / 212 channels, whose
    NHWC rows are not 16-byte multiples, keep the CUDA-core kernels."""
    rows = _dispatch(models.Cond_SRVAE(cr, 64))
    for net, kind, ci, co, h, f, d, wl in rows:
        if ci % 8 == 0 and co % 8 == 0 and min(ci, co) >= 16:
            assert (f, d, wl) == (1, 1, 1), (net, kind, ci, co, h, f, d, wl)
        if ci % 8 or co % 8:
            assert (ci if ci % 8 else co) in (4, 42, 84, 53, 106, 212), (net, kind, ci, co)     # 4: the image layers
            assert wl == 0 and (f == 0 or ci % 8 == 0) and (d == 0 or co % 8 == 0), (net, kind, ci, co, h, f, d, wl)
    keys = {r[:5] for r in rows}
    for m in MOVED[cr]:
        assert m in keys, m
        r = [x for x in rows if x[:5] == m][0]
        assert r[5:] == (1, 1, 1), r


@pytest.mark.parametrize("C", [42, 84, 53, 106, 212, 8, 4, 12, 20])
def test_channel_rule(C):
    """C % 8 != 0 (rows that are not 16-byte multiples) and C = 8 stay on the CUDA-core kernels, as reduction, as output
    of the weight gradient and as its X operand; every other multiple of 8 from 24 up runs on tcgen05."""
    for H in (4, 8, 16):
        assert lib.tc_would_run(BF16, C, 64, H, H) == 0
        assert lib.conv2d_wgrad_layout(BF16, 2, H, H, 64, C, 3) == 0        # Ca = C
        assert lib.conv2d_wgrad_layout(BF16, 2, H, H, C, 64, 3) == 0        # Cb = C
        assert lib.convT2d_wgrad_layout(BF16, 2, H, H, C, 64) == 0          # Ca = C
        assert lib.convT2d_wgrad_layout(BF16, 2, H, H, 64, C) == 0          # Cb = C


@pytest.mark.parametrize("C", [24, 40, 56, 72, 88, 104, 120, 168, 336, 424, 672, 848, 1344, 1696])
def test_ragged_channels_accepted(C):
    for H in (4, 8):
        assert lib.tc_would_run(BF16, C, 64, H, H) == 1
        assert lib.tc_would_run(BF16, 64, C, H, H) == 1
        assert lib.conv2d_wgrad_layout(BF16, 2, H, H, 64, C, 3) == 1
        assert lib.conv2d_wgrad_layout(BF16, 2, H, H, C, 64, 3) == 1
        assert lib.conv2d_wgrad_layout(BF16, 2, 2 * H, 2 * H, C, C, 4) == 1
        assert lib.convT2d_wgrad_layout(BF16, 2, H, H, C, 64) == 1
        assert lib.convT2d_wgrad_layout(BF16, 2, H, H, 64, C) == 1
        assert lib.tc_would_run(F32, C, 64, H, H) == 0                              # fp32 parity mode stays on CUDA cores
        assert lib.conv2d_wgrad_layout(F32, 2, H, H, 64, C, 3) == 0
