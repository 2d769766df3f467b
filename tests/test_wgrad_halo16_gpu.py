"""Weight and bias gradients of the 3x3 stride-1 convs that produce 16 channels (64 -> 16, 16 -> 16) on the tcgen05 halo
kernel (wgrad_halo.cu), through svrs_conv2d_wgrad, against float64 on the CPU.

Covers the benchmarked steps' shapes (64x64, 32x32 and 16x16 maps at 128 patches), several pixel splits (the split count
follows the batch), ragged splits (the last split owns fewer pixel steps), both gradient layouts (torch layout with fp32
atomics, and the packed [tap][Cin][Cout] layout the fused optimiser reads), a NULL bias gradient, and a map that does not
tile into 8 x 16 pixels (served by wgrad_tc).  Every output sits inside a sentinel guard band."""
import pytest
import torch

from helpers import BF16, Guarded, lib, nhwc, report, st

pytestmark = pytest.mark.gpu
DEV = "cuda"
RTOL = 1e-5     # weight-gradient bound of the repo: max |err| relative to max |ref|

CASES = [
    # N, H, W, Cin   (Cout = 16)
    (128, 64, 64, 64), (128, 64, 64, 16),       # decoder_x tail
    (128, 32, 32, 64), (128, 32, 32, 16),       # decoder_y tail
    (128, 16, 16, 16),                          # first conv of the second down_blocks
    (1, 64, 64, 64), (2, 32, 32, 16),           # few pixel steps: small splits
    (7, 16, 24, 16), (7, 16, 24, 64),           # 21 pixel steps in 5 splits of <= 5 steps (ragged last split)
    (3, 48, 16, 64),                            # non-square map
    (5, 8, 16, 16), (2, 12, 32, 64),            # maps that do not tile into 8 x 16 pixels: wgrad_tc
]


def _ref(N, H, W, Cin, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(N, Cin, H, W, generator=g).to(torch.bfloat16)
    gy = torch.randn(N, 16, H, W, generator=g).to(torch.bfloat16)
    dw = torch.nn.grad.conv2d_weight(x.double(), (16, Cin, 3, 3), gy.double(), padding=1)
    return x, gy, dw, gy.double().sum(dim=(0, 2, 3))


@pytest.mark.parametrize("packed", [False, True])
@pytest.mark.parametrize("case", CASES)
def test_wgrad16_layers_against_fp64(case, packed):
    N, H, W, Cin = case
    x, gy, dwr, dbr = _ref(N, H, W, Cin, sum(case) + 11)
    xd, gyd = nhwc(x.to(DEV), torch.bfloat16), nhwc(gy.to(DEV), torch.bfloat16)
    layout = lib.conv2d_wgrad_layout(BF16, N, H, W, Cin, 16, 3)
    assert layout == 1, "the tcgen05 kernels (halo, or wgrad_tc off the 8 x 16 tiling) take every 16-channel layer"
    dw = Guarded((16, Cin, 3, 3), torch.float32, fill=0.0)
    dwp = Guarded((9, Cin, 16), torch.float32, fill=0.0)
    db = Guarded((16,), torch.float32, fill=0.0)
    for _ in range(2):      # the kernels accumulate: two calls give twice the gradient
        lib.conv2d_wgrad(xd.data_ptr(), gyd.data_ptr(), dw.t.data_ptr(), dwp.t.data_ptr() if packed else None, db.t.data_ptr(),
                         BF16, N, H, W, Cin, 16, 3, 0, st())
    torch.cuda.synchronize()
    if packed:
        got = dwp.t.permute(2, 1, 0).reshape(16, Cin, 3, 3)
        assert bool((dw.t == 0).all()), "the packed route must not touch the torch-layout buffer"
    else:
        got = dw.t
    report(f"wgrad16 {case} packed={packed} dw", got, 2 * dwr, RTOL)
    report(f"wgrad16 {case} packed={packed} db", db.t, 2 * dbr, RTOL)
    assert dw.intact() and dwp.intact() and db.intact(), "write outside an output buffer"


@pytest.mark.parametrize("case", [(128, 64, 64, 64), (7, 16, 24, 16)])
def test_wgrad16_halo_without_bias(case):
    """db = NULL: the weight gradient alone, and nothing written to a bias buffer placed next to it."""
    N, H, W, Cin = case
    x, gy, dwr, _ = _ref(N, H, W, Cin, sum(case) + 3)
    xd, gyd = nhwc(x.to(DEV), torch.bfloat16), nhwc(gy.to(DEV), torch.bfloat16)
    dwp = Guarded((9, Cin, 16), torch.float32, fill=0.0)
    dw = Guarded((16, Cin, 3, 3), torch.float32, fill=0.0)
    lib.conv2d_wgrad(xd.data_ptr(), gyd.data_ptr(), dw.t.data_ptr(), dwp.t.data_ptr(), None, BF16, N, H, W, Cin, 16, 3, 0, st())
    torch.cuda.synchronize()
    report(f"wgrad16 {case} no bias dw", dwp.t.permute(2, 1, 0).reshape(16, Cin, 3, 3), dwr, RTOL)
    assert bool((dw.t == 0).all()) and dw.intact() and dwp.intact()
