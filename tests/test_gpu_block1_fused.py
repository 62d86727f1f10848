"""Fused block1.2 -> block1.3 + skip1 tcgen05 kernel (csrc/block1_tc.cu) against the oracle and, bit for bit, against the
two-kernel tensor-core path it replaces."""
import contextlib

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from oracle import xfeat_oracle as orc  # noqa: E402


@pytest.fixture(scope="module")
def xf():
    from accelerated_features_b200 import XFeat
    return XFeat()


@contextlib.contextmanager
def block1_fused(xf, on):
    old = xf._lib.xfeat_get_block1_fused()
    xf._lib.xfeat_set_block1_fused(on)
    try:
        yield
    finally:
        xf._lib.xfeat_set_block1_fused(old)


def relerr(a, b):
    return float((a.double() - b.double()).abs().max() / (b.double().abs().max() + 1e-30))


def block1_tail(xf, a2, xn, fused):
    """a2 (B,8,H/2,W/2), xn (B,1,H,W) CPU tensors -> x1s (B,24,H/4,W/4) from xfeat_debug_block1_tail."""
    from accelerated_features_b200 import _lib
    B, _, H, W = xn.shape
    a2d = a2.permute(0, 2, 3, 1).contiguous().cuda()
    xnd = xn[:, 0].contiguous().cuda()
    out = torch.full((B, H // 4, W // 4, 24), float("nan"), device="cuda")
    scratch = torch.empty(B * (H // 2) * (W // 2) * 64, dtype=torch.uint8, device="cuda")
    with block1_fused(xf, fused):
        assert xf._lib.xfeat_get_block1_fused() == fused
        _lib.check(xf._lib.xfeat_debug_block1_tail(xf._ctx, a2d.data_ptr(), xnd.data_ptr(), B, H, W, out.data_ptr(),
                                                   scratch.data_ptr(), scratch.numel(), torch.cuda.current_stream().cuda_stream),
                   "block1 tail")
        torch.cuda.synchronize()
    return out.permute(0, 3, 1, 2).cpu()


# (B, H, W) of the full-resolution image: VGA, the two star scales, 800x576, the 32x32 minimum, and 148x268 -- quarter-res
# 37 x 67, primes larger than any tile side the tile picker allows (TQH * (TQW + 1) <= 128, TQW <= 62) other than a single
# row, so the last tile is ragged in both directions.
CASES = [(3, 480, 640), (3, 576, 768), (3, 1248, 1664), (3, 576, 800), (3, 32, 32), (2, 148, 268)]


@pytest.mark.parametrize("case", CASES, ids=lambda c: f"B{c[0]}_{c[1]}x{c[2]}")
def test_block1_tail_vs_oracle_and_unfused(xf, oracle_state, case):
    B, H, W = case
    sd = oracle_state
    g = torch.Generator().manual_seed(H * 7 + W)
    a2 = torch.relu(torch.randn(B, 8, H // 2, W // 2, generator=g) * 2.0)   # block1.1 outputs are post-ReLU
    xn = torch.randn(B, 1, H, W, generator=g)
    t = orc._basic_layer(sd, "block1.2", a2, 1)
    want = orc._basic_layer(sd, "block1.3", t, 2) + F.conv2d(F.avg_pool2d(xn, 4, stride=4), sd["skip1.1.weight"], sd["skip1.1.bias"])
    fused = block1_tail(xf, a2, xn, 1)
    err = relerr(fused, want)
    print(f"block1 fused {B}x{H}x{W}: rel err {err:.2e}")
    assert err < 1e-5, err
    two_kernel = block1_tail(xf, a2, xn, 0)
    assert torch.equal(fused, two_kernel)


def test_block1_fused_is_default(xf):
    assert xf._lib.xfeat_get_block1_fused() == 1
