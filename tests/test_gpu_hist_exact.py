"""k5_hist's sparse histograms byte for byte against a numpy restatement built on the oracle's BGR -> HSV.

tsd_hist_sparse runs the chain's histogram kernel on device-resident windows and returns everything later stages read: the entries
(bin << 16 | count in bin order, zero padded), the per-window moments (s1 and s11 summed lane by lane in rank order, then by the
warp's xor shuffle tree), A, sqrt(A), a, nnz, the pixel hash, the 25 group energy bounds and the chunk starts k5_gram walks.
The windows are random, smooth, flat (one bin holding more than 255 pixels), single-colour, grey (d = 0) and built from a few
channel values (ties between the maximum channels), at D = 25 (640-pixel kernel) and D = 32 (1024-pixel kernel), in the packed
public layout (3 D^2 bytes apart: byte loads and, for windows that happen to start on a 4-byte boundary, word loads) and in the
chain's padded layout (a multiple of 16 bytes apart: staged through shared memory), the padding filled with non-zero bytes.
"""
import numpy as np
import pytest

K1, K2 = np.uint32(0x9E3779B1), np.uint32(0x85EBCA6B)
META = np.dtype([("s1", "<f8"), ("s11", "<f8"), ("A", "<f8"), ("rA", "<f8"), ("a", "<f4"), ("nnz", "<i4"), ("hash", "<u4"), ("pad", "<u4")])
ROWS = 28                       # 25 group energies + 3 rows of chunk starts


def make_windows(D, n, seed):
    rng = np.random.default_rng(seed)
    w = rng.integers(0, 256, (n, D, D, 3), dtype=np.uint8)                        # random
    k = n // 8
    y, x = np.mgrid[0:D, 0:D]
    for i in range(k, 2 * k):                                                      # smooth: few distinct bins
        c = rng.integers(0, 256, 3)
        g = rng.integers(-4, 5, (2, 3))
        w[i] = np.clip(c + y[..., None] * g[0] + x[..., None] * g[1], 0, 255)
    for i in range(2 * k, 3 * k):                                                  # flat: one bin > 255 pixels, a few others
        w[i] = rng.integers(0, 256, 3)
        m = rng.random((D, D)) < 0.1
        w[i][m] = rng.integers(0, 256, (int(m.sum()), 3))
    for i in range(3 * k, 4 * k):                                                  # single colour
        w[i] = rng.integers(0, 256, 3)
    for i in range(4 * k, 5 * k):                                                  # grey: b = g = r
        w[i] = rng.integers(0, 256, (D, D, 1))
    for i in range(5 * k, 6 * k):                                                  # three channel values: ties of the maximum
        w[i] = rng.choice(np.array([0, 1, 128, 254, 255], np.uint8), (D, D, 3))
    w[6 * k] = 0
    w[6 * k + 1] = 255
    return w


def reference(windows, oracle):
    n, D = windows.shape[0], windows.shape[1]
    npx, es = D * D, (D * D + 3) & ~3
    px = windows.reshape(n, npx, 3)
    hsv = oracle.bgr2hsv(px.reshape(1, -1, 3)).reshape(n, npx, 3).astype(np.int64)
    bins = (hsv[..., 0] * 50 // 180) * 60 + hsv[..., 1] * 60 // 256                # calcHist([0,1], [50,60], [0,180,0,256])
    bgr = px[..., 0].astype(np.uint32) | (px[..., 1].astype(np.uint32) << 8) | (px[..., 2].astype(np.uint32) << 16)
    x = bgr * K1 + np.arange(npx, dtype=np.uint32) * K2
    hashes = ((x ^ (x >> np.uint32(15))).astype(np.uint64).sum(axis=1) & 0xffffffff).astype(np.uint32)
    ent = np.zeros((n, es), np.uint32)
    meta = np.zeros(n, META)
    energies = np.zeros((ROWS, n), np.float32)
    for i in range(n):
        counts = np.bincount(bins[i], minlength=3000)
        occ = np.nonzero(counts)[0]
        c = counts[occ].astype(np.uint32)
        nnz = len(occ)
        ent[i, :nnz] = (occ.astype(np.uint32) << 16) | c
        a = np.float32(1.0 / float(c.max()))
        h = (c.astype(np.float32) * a).astype(np.float64)
        hp = np.zeros((nnz + 31) // 32 * 32)
        hp[:nnz] = h
        s1, s11 = np.zeros(32), np.zeros(32)
        for row in hp.reshape(-1, 32):                                              # lane l sums ranks l, l + 32, ... in order
            s1 = s1 + row
            s11 = s11 + row * row
        for o in (16, 8, 4, 2, 1):                                                  # v += shfl_xor(v, o)
            s1 = s1 + s1[np.arange(32) ^ o]
            s11 = s11 + s11[np.arange(32) ^ o]
        A = s11[0] - s1[0] * s1[0] * (1.0 / 3000.0)
        meta[i] = (s1[0], s11[0], A, np.sqrt(A), a, nnz, hashes[i], 0)
        gsum = np.zeros(25, np.uint64)
        np.add.at(gsum, occ // 120, c.astype(np.uint64) ** 2)
        energies[:25, i] = a * np.sqrt(gsum.astype(np.float32)) * np.float32(1.00001)
        pf = [int(np.searchsorted(occ, 512 * ch)) for ch in (1, 2, 3, 4, 5)] + [nnz]
        energies[25:, i] = np.array([pf[0] | pf[1] << 16, pf[2] | pf[3] << 16, pf[4] | pf[5] << 16], np.uint32).view(np.float32)
    return ent, meta, energies


@pytest.mark.gpu
@pytest.mark.parametrize("D", [25, 32])
@pytest.mark.parametrize("layout", ["packed", "padded"])
def test_hist_sparse_exact(oracle, D, layout):
    import torch
    import tsd_b200
    n = 1000
    win = make_windows(D, n, seed=D * 7 + (layout == "padded"))
    ws = 3 * D * D if layout == "packed" else (3 * D * D + 15) & ~15
    buf = np.full((n, ws), 0xA5, np.uint8)                                          # non-zero padding: pad pixels must not count
    buf[:, :3 * D * D] = win.reshape(n, -1)
    es = (D * D + 3) & ~3
    dev = torch.device("cuda", 0)
    d_win = torch.from_numpy(buf).to(dev)
    d_ent = torch.full((n, es), 0x7777, dtype=torch.int32, device=dev)
    d_meta = torch.zeros((n, 48), dtype=torch.uint8, device=dev)
    d_en = torch.zeros((ROWS, n), dtype=torch.float32, device=dev)
    with tsd_b200.Context(0, "det") as ctx:
        ctx.hist_sparse(d_win.data_ptr(), n, D, ws, d_ent.data_ptr(), d_meta.data_ptr(), d_en.data_ptr())
        ctx.synchronize()
    ent, meta, energies = reference(win, oracle)
    got_ent = d_ent.cpu().numpy().view(np.uint32)
    got_meta = d_meta.cpu().numpy().reshape(-1).view(META)
    got_en = d_en.cpu().numpy()
    for i in range(n):
        nnz = int(meta[i]["nnz"])
        assert np.array_equal(got_ent[i, :(nnz + 3) & ~3], ent[i, :(nnz + 3) & ~3]), "entries of window %d" % i
    assert got_meta.tobytes() == meta.tobytes()
    assert got_en.tobytes() == energies.tobytes()
    # a count above 255 and a grey window (a single entry, in bin 0) are among them
    assert (ent & 0xffff).max() > 255
    assert any(meta["nnz"][i] == 1 and ent[i, 0] >> 16 == 0 for i in range(n))


def test_hist_reference_regimes(oracle):
    """The windows reach the regimes the GPU test names (CPU)."""
    win = make_windows(25, 200, seed=1)
    ent, meta, energies = reference(win, oracle)
    assert (ent & 0xffff).max() > 255
    assert (meta["nnz"] == 1).sum() >= 25
    assert meta["nnz"].max() > 256
    px = win.reshape(-1, 3).astype(int)
    v = px.max(axis=1)
    for ch in range(3):
        assert (px[:, ch] == v).any()


def test_bin_rule_every_colour(oracle):
    """The integer rule k5_hist bins a pixel with (OpenCV's RGB2HSV_b division tables, hue bin (H * 18205) >> 16, saturation bin
    (S * 60) >> 8) against the oracle's BGR -> HSV and calcHist's bins, for all 2^24 BGR values (CPU)."""
    i = np.arange(1, 256)
    sdiv = np.concatenate([[0], np.rint((255 << 12) / (1.0 * i))]).astype(np.int64)          # lrint: half to even, as np.rint
    hdiv = np.concatenate([[0], np.rint((180 << 12) / (6.0 * i))]).astype(np.int64)
    c = np.arange(1 << 24, dtype=np.uint32)
    b, g, r = (c & 255).astype(np.int64), ((c >> 8) & 255).astype(np.int64), (c >> 16).astype(np.int64)
    v, m = np.maximum(b, np.maximum(g, r)), np.minimum(b, np.minimum(g, r))
    d = v - m
    h = np.where(v == r, g - b, np.where(v == g, b - r + 2 * d, r - g + 4 * d))
    S = (d * sdiv[v] + (1 << 11)) >> 12
    h = (h * hdiv[d] + (1 << 11)) >> 12
    H = np.where(h < 0, h + 180, h)
    kernel = ((H * 18205) >> 16) * 60 + ((S * 60) >> 8)
    bgr = np.stack([b, g, r], axis=1).astype(np.uint8)
    hsv = oracle.bgr2hsv(bgr.reshape(1, -1, 3)).reshape(-1, 3).astype(np.int64)
    ref = (hsv[:, 0] * 50 // 180) * 60 + hsv[:, 1] * 60 // 256
    assert H.max() < 180 and np.array_equal(kernel, ref)
