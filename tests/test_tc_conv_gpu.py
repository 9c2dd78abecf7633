"""tcgen05 implicit-GEMM convolution vs the fp32 CUDA-core kernel on the same seeded data (per layer).
Operands are fp16-exact weights and split-fp16 (hi+lo) or plain fp16 activations; the reference result is computed
in fp32 from exactly the values the tensor path sees, so the tolerance only covers fp32 accumulation order and the
output rounding (split: ~2^-22 relative; plain fp16 output: 2^-11 relative)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _data(cin, cout, h, w, kk, seed=0):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((cin, h, w), dtype=np.float32)
    wgt = (rng.standard_normal((cout, cin, kk), dtype=np.float32) / np.sqrt(cin * 9)).astype(np.float32)
    b = rng.standard_normal(cout).astype(np.float32) * 0.1
    res = rng.standard_normal((cout, h, w), dtype=np.float32)
    return x, wgt, b, res


def _check(o_tc, o_ref, split):
    err = np.abs(o_tc - o_ref)
    scale = np.abs(o_ref).max() + 1e-6
    tol = (2e-5 if split else 2e-3) * scale
    bad = np.argwhere(err > tol)
    return float(err.max()), float(tol), bad


@pytest.mark.parametrize("c", [64, 96, 128, 192])
@pytest.mark.parametrize("split", [1, 0])
def test_conv3x3_res_leaky(pkg, c, split):
    h, w = 21, 70  # 2 column tiles (62 + 8) and a ragged last row tile
    x, wgt, b, res = _data(c, c, h, w, 9, seed=c)
    o_tc, o_ref = pkg.selftest_conv(0, x, wgt, b, res=res, slope=0.2, split=bool(split))
    mx, tol, bad = _check(o_tc, o_ref, split)
    assert len(bad) == 0, "max err %g (tol %g); first bad idx %s of %d" % (mx, tol, bad[:5].tolist(), len(bad))


@pytest.mark.parametrize("c", [32, 48, 64, 96, 128, 192])
@pytest.mark.parametrize("split", [1, 0])
def test_conv3x3_self_residual(pkg, c, split):
    """Residual == the conv's own input (the ResConv blocks): the kernel adds it on the tensor core through an identity
    tap instead of reading it in the epilogue; passing res=x selects that path."""
    h, w = 21, 70
    x, wgt, b, _ = _data(c, c, h, w, 9, seed=100 + c)
    x = np.ascontiguousarray(x, np.float32)
    o_tc, o_ref = pkg.selftest_conv(0, x, wgt, b, res=x, slope=0.2, split=bool(split))
    mx, tol, bad = _check(o_tc, o_ref, split)
    assert len(bad) == 0, "max err %g (tol %g); first bad idx %s of %d" % (mx, tol, bad[:5].tolist(), len(bad))


@pytest.mark.parametrize("cin", [64, 96, 128, 192])
@pytest.mark.parametrize("split", [1, 0])
def test_flow_head_deconv_five_planes(pkg, cin, split):
    """deconv4x4s2 (24 channels) + PixelShuffle(2) keeping the five planes the flow / mask update reads."""
    h, w = 9, 70
    x, wgt, b, _ = _data(cin, 24, h, w, 16, seed=cin + 5)
    o_tc, o_ref = pkg.selftest_conv(3, x, wgt, b, split=bool(split), ps=2)
    mx, tol, bad = _check(o_tc[:5], o_ref[:5], split)
    assert len(bad) == 0, "max err %g (tol %g); first bad idx %s of %d" % (mx, tol, bad[:5].tolist(), len(bad))
    assert not o_tc[5].any()


def test_conv3x3_single_taps(pkg):
    """One non-zero tap at a time: localises a wrong shared-memory view (row/column shift) to its (dy,dx)."""
    c, h, w = 64, 10, 64
    x, wgt, b, _ = _data(c, c, h, w, 9, seed=7)
    report = []
    for tap in range(9):
        wt = np.zeros_like(wgt)
        wt[:, :, tap] = wgt[:, :, tap]
        o_tc, o_ref = pkg.selftest_conv(0, x, wt, b * 0, res=None, slope=1.0, split=True)
        mx, tol, bad = _check(o_tc, o_ref, 1)
        report.append((tap, mx, len(bad)))
    assert all(n == 0 for _, _, n in report), report


@pytest.mark.parametrize("cin,cout,ps", [(64, 24, 2), (192, 24, 2), (96, 5, 1)])
def test_deconv_pixelshuffle(pkg, cin, cout, ps):
    h, w = 9, 70
    x, wgt, b, _ = _data(cin, cout, h, w, 16, seed=cin + cout)
    o_tc, o_ref = pkg.selftest_conv(1, x, wgt, b, split=True, ps=ps)
    mx, tol, bad = _check(o_tc, o_ref, 1)
    assert len(bad) == 0, "max err %g (tol %g); first bad idx %s of %d" % (mx, tol, bad[:5].tolist(), len(bad))


@pytest.mark.parametrize("cin,cout", [(12, 32), (7, 96), (12, 48), (32, 64), (48, 96), (64, 128), (96, 192)])
def test_conv3x3_stride2(pkg, cin, cout):
    """Stride-2 conv over the space-to-depth input (block-head convs: narrow fp32-critical inputs padded to 16 ch)."""
    h, w = 44, 140  # output 22 x 70: two column tiles, ragged rows
    x, wgt, b, _ = _data(cin, cout, h, w, 9, seed=cin * 7 + cout)
    o_tc, o_ref = pkg.selftest_conv(2, x, wgt, b, slope=0.2, split=True)
    mx, tol, bad = _check(o_tc, o_ref, 1)
    assert len(bad) == 0, "max err %g (tol %g); first bad idx %s of %d" % (mx, tol, bad[:5].tolist(), len(bad))


@pytest.mark.parametrize("split", [1, 0])
@pytest.mark.parametrize("self_res", [True, False])
@pytest.mark.parametrize("h,w", [(11, 140), (4, 126), (5, 127), (9, 300)])
def test_conv3x3_n64_ragged_tiles(pkg, h, w, self_res, split):
    """N = 64 on the paired whole-chunk issue path (tiles of 8 rows x 62 columns): several column tiles, ragged last column
    and row tiles, the self-residual identity tap and the epilogue residual."""
    c = 64
    x, wgt, b, res = _data(c, c, h, w, 9, seed=h * 1000 + w)
    x = np.ascontiguousarray(x, np.float32)
    o_tc, o_ref = pkg.selftest_conv(0, x, wgt, b, res=x if self_res else res, slope=0.2, split=bool(split))
    mx, tol, bad = _check(o_tc, o_ref, split)
    assert len(bad) == 0, "max err %g (tol %g); first bad idx %s of %d" % (mx, tol, bad[:5].tolist(), len(bad))


@pytest.mark.parametrize("c", [48, 96, 128, 192])
@pytest.mark.parametrize("split", [1, 0])
def test_conv5x5_row_stages(pkg, c, split):
    """5x5 stride-1 pad-2 convolution (the residual blocks of the rife / HD / UHD / anime flownets) on the tensor cores: one
    kernel row (five shifted views of 2*MT image rows) per pipeline stage; two column tiles (60 + 10), ragged last row tile."""
    h, w = 21, 70
    rng = np.random.default_rng(c)
    x = rng.standard_normal((c, h, w), dtype=np.float32)
    wgt = (rng.standard_normal((c, c, 25), dtype=np.float32) / np.sqrt(c * 25)).astype(np.float32)
    b = rng.standard_normal(c).astype(np.float32) * 0.1
    res = rng.standard_normal((c, h, w), dtype=np.float32)
    o_tc, o_ref = pkg.selftest_conv(4, x, wgt, b, res=res, slope=0.2, split=bool(split))
    mx, tol, bad = _check(o_tc, o_ref, split)
    assert len(bad) == 0, "max err %g (tol %g); first bad idx %s of %d" % (mx, tol, bad[:5].tolist(), len(bad))


def test_conv5x5_single_taps(pkg):
    """One non-zero tap at a time localises a wrong view (row stage dy / column shift dx)."""
    c, h, w = 48, 10, 64
    rng = np.random.default_rng(11)
    x = rng.standard_normal((c, h, w), dtype=np.float32)
    wgt = (rng.standard_normal((c, c, 25), dtype=np.float32) / np.sqrt(c)).astype(np.float32)
    report = []
    for tap in (0, 4, 7, 12, 20, 24):
        wt = np.zeros_like(wgt)
        wt[:, :, tap] = wgt[:, :, tap]
        o_tc, o_ref = pkg.selftest_conv(4, x, wt, np.zeros(c, np.float32), res=None, slope=1.0, split=True)
        mx, tol, bad = _check(o_tc, o_ref, 1)
        report.append((tap, mx, len(bad)))
    assert all(n == 0 for _, _, n in report), report
