"""CPU replay of the tcgen05 conv's operand views (csrc/tc_conv.cu): a numpy model of the no-swizzle K-major shared-memory
descriptors (row i of an operand = 16 contiguous bytes at start + i*16, second K half LBO bytes further) applied to
(a) the real packed weights (rife_b200_debug_pack_weights) and (b) a halo tile laid out as TMA delivers it, with the
exact start-address / TMEM-column arithmetic of the kernel's issue loops.  The unpaired issue order is the one verified
on the GPU (tests/test_tc_conv_gpu.py); the paired order of umma_issue_chunk_paired (tools/gen_mma_issue.py chunk_block:
per kernel column dx the paired rows -- one 2N-column MMA feeds the dy=2 tap of accumulator j-1 and the dy=0 tap of
accumulator j -- then the dy=1 taps; the identity tap comes last and is not replayed here) must produce the same
accumulators, and both must equal a direct 3x3 convolution / 4x4 stride-2 deconvolution of the tile.
The generated issue code itself must be what tools/gen_mma_issue.py produces."""
import ctypes
import importlib.util
import os

import numpy as np
import pytest

TWP = 64


def _pack(pkg, mode, w, cout, cin, N, ocs, paired):
    L = pkg.lib()
    n = (cin // 16) * 9 * 2 * N * 8
    out = np.zeros(n, np.uint16)
    w = np.ascontiguousarray(w, np.float32)
    r = L.rife_b200_debug_pack_weights(mode, cout, cin, N, ocs, paired, w.ctypes.data, out.ctypes.data, n)
    assert r == 0
    return out.view(np.float16).astype(np.float32)


def _a_view(slab, rows, start16):
    """A operand (128 x 16) from one K chunk's slab [2 halves][rows][64 px][8]: row i = pixel start16 + i of each half."""
    flat = slab.reshape(2, rows * TWP, 8)
    pad = np.zeros((2, 128 + 4 * TWP, 8), np.float32)  # overrun pad behind the slab (zeros here; those rows are halo columns)
    flat = np.concatenate([flat, pad], axis=1)
    return np.concatenate([flat[0, start16:start16 + 128], flat[1, start16:start16 + 128]], axis=1)  # [128][16]


def _b_view(wchunk, start16, lbo16, n):
    """B operand (n x 16): row r = 16 B at (start16 + r), second K half lbo16 rows further; wchunk = fp16 values of one K chunk"""
    rows = wchunk.reshape(-1, 8)
    return np.concatenate([rows[start16:start16 + n], rows[start16 + lbo16:start16 + lbo16 + n]], axis=1)  # [n][16]


def _accumulate(slabs, wpk, N, MT, paired):
    """Replays the mainloop of one tile: returns acc [MT][128][N]"""
    rows = 2 * MT + 2
    kcs = len(slabs)
    acc = np.zeros((128, MT * N), np.float64)
    wk = wpk.reshape(kcs, -1)
    rowstep = 2 * TWP
    for kc in range(kcs):
        slab = slabs[kc]
        if not paired:
            for tap in range(9):
                dy, dx = divmod(tap, 3)
                B = _b_view(wk[kc], tap * 2 * N, N, N)
                for m in range(MT):
                    A = _a_view(slab, rows, dy * TWP + dx + m * rowstep)
                    acc[:, m * N:(m + 1) * N] += A @ B.T
        else:
            for dx in range(3):
                blk = dx * 2 * 3 * N  # 16-byte rows from the chunk start
                for j in range(MT + 1):  # even views: paired rows
                    A = _a_view(slab, rows, dx + j * rowstep)
                    if j == 0:
                        acc[:, 0:N] += A @ _b_view(wk[kc], blk + N, 3 * N, N).T
                    elif j == MT:
                        acc[:, (MT - 1) * N:MT * N] += A @ _b_view(wk[kc], blk, 3 * N, N).T
                    else:
                        acc[:, (j - 1) * N:(j + 1) * N] += A @ _b_view(wk[kc], blk, 3 * N, 2 * N).T
                for m in range(MT):  # odd views (one row down, dy = 1 rows of the block)
                    A = _a_view(slab, rows, dx + TWP + m * rowstep)
                    acc[:, m * N:(m + 1) * N] += A @ _b_view(wk[kc], blk + 2 * N, 3 * N, N).T
    return acc.reshape(128, MT, N).transpose(1, 0, 2)


def _tile(cin, MT, rng):
    rows = 2 * MT + 2
    x = rng.standard_normal((cin, rows, TWP)).astype(np.float16).astype(np.float32)  # halo tile, planar
    slabs = [x[kc * 16:(kc + 1) * 16].reshape(2, 8, rows, TWP).transpose(0, 2, 3, 1).copy() for kc in range(cin // 16)]
    return x, slabs


@pytest.mark.parametrize("cin,cout,N,MT", [(64, 64, 64, 4), (32, 32, 32, 4), (96, 96, 96, 2), (128, 128, 128, 2), (48, 40, 48, 4)])
def test_conv3x3_views_paired_equals_unpaired_equals_direct(pkg, cin, cout, N, MT):
    rng = np.random.default_rng(cin * 7 + N)
    w = (rng.standard_normal((cout, cin, 3, 3)) * 0.1).astype(np.float16).astype(np.float32)
    x, slabs = _tile(cin, MT, rng)
    ref = np.zeros((MT, 128, N))
    for m in range(MT):  # position p of accumulator m: output row 2m + p // 64 (tile rows), column p % 64 (valid < 62)
        for p in range(128):
            r, c = 2 * m + p // TWP, p % TWP
            if c >= TWP - 2:
                continue
            patch = x[:, r:r + 3, c:c + 3]  # halo tile coordinates: output (r, c) reads rows r..r+2, cols c..c+2
            ref[m, p, :cout] = np.tensordot(w, patch, axes=([1, 2, 3], [0, 1, 2]))
    valid = (np.arange(128) % TWP) < TWP - 2
    for paired in (0, 1):
        acc = _accumulate(slabs, _pack(pkg, 0, w, cout, cin, N, 0, paired), N, MT, bool(paired))
        assert np.allclose(acc[:, valid], ref[:, valid], atol=1e-3), (paired, np.abs(acc[:, valid] - ref[:, valid]).max())


def test_deconv_views_paired_equals_unpaired(pkg):
    """deconv4x4 s2 as a 3x3-neighbourhood GEMM with N = 4 parities x ocs columns (flow head: 24 -> N = 96)"""
    cin, cout, ocs, N, MT = 64, 24, 24, 96, 2
    rng = np.random.default_rng(5)
    w = (rng.standard_normal((cout, cin, 4, 4)) * 0.1).astype(np.float16).astype(np.float32)
    x, slabs = _tile(cin, MT, rng)
    a0 = _accumulate(slabs, _pack(pkg, 1, w, cout, cin, N, ocs, 0), N, MT, False)
    a1 = _accumulate(slabs, _pack(pkg, 1, w, cout, cin, N, ocs, 1), N, MT, True)
    valid = (np.arange(128) % TWP) < TWP - 2
    assert np.allclose(a0[:, valid], a1[:, valid], atol=1e-3)
    # direct: out(2y+py, 2x+px, oc) = sum_{ic, ky, kx} in(iy, ix) w[oc][ic][ky][kx] with 2*iy - 1 + ky = 2y+py (ncnn deconvolution, pad 1)
    m, p = 1, 70
    r, c = 2 * m + p // TWP, p % TWP  # input pixel (y, x) = halo (r + 1, c + 1)
    for par in range(4):
        py, px = par >> 1, par & 1
        for oc in range(cout):
            s = 0.0
            for ky in range(4):
                for kx in range(4):
                    ty, tx = 2 * (r + 1) + py + 1 - ky, 2 * (c + 1) + px + 1 - kx
                    if ty % 2 or tx % 2:
                        continue
                    s += float(np.dot(x[:, ty // 2, tx // 2], w[oc, :, ky, kx]))
            assert abs(a1[m, p, par * ocs + oc] - s) < 1e-3, (par, oc, a1[m, p, par * ocs + oc], s)


def test_pack_weights_rejects_unknown_layout(pkg):
    """paired is -1 (the kernel's layout for this N), 0 or 1; anything else is an argument error."""
    w = np.zeros((16, 16, 3, 3), np.float32)
    out = np.zeros(9 * 2 * 16 * 8, np.uint16)
    for paired in (-2, 2, 3):
        assert pkg.lib().rife_b200_debug_pack_weights(0, 16, 16, 16, 0, paired, w.ctypes.data, out.ctypes.data, out.size) != 0, paired
    assert pkg.lib().rife_b200_debug_pack_weights(0, 16, 16, 16, 0, -1, w.ctypes.data, out.ctypes.data, out.size) == 0


def test_generated_mma_issue_is_current(tmp_path):
    """csrc/tc_mma_issue.inc is the output of tools/gen_mma_issue.py (an edit of either alone does not pass)."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("gen_mma_issue", os.path.join(root, "tools", "gen_mma_issue.py"))
    gen = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gen)
    out = tmp_path / "tc_mma_issue.inc"
    gen.main(str(out))
    assert out.read_text() == open(os.path.join(root, "rife-ncnn-vulkan_b200", "csrc", "tc_mma_issue.inc")).read()
