"""CPU: the index logic of the power-of-two pyramid kernels (csrc/farneback.cu: HalfPyr, pyr_vsweep_kernel,
pyr_hpass_kernel, pyr_hpass1_kernel), restated with Python loops and checked against the oracle's own blur + resize.

1. The constants the kernels are specialised on (stride S = 2^l, taps T, window start S * d - NB) are what the
   collapsed blur + resize filter of a pyr_scale 0.5 level IS, derived from oracle/farneback_np's resize coefficients
   and blur parameters (farneback.cu: farneback_setup makes the same check on its tables at mavd_create and falls
   back per level and axis).
2. The polyphase schedule of the sweep — which (output row, tap) a source row feeds in which of the <= 3 live
   accumulators, when an output is finished, which band stores it — gives every output row of every level exactly
   its T taps, in ascending order, from the REFLECT_101 rows, once.
3. The whole restatement (sweep with level 1's horizontal pass inside, vectorised horizontal passes above) reproduces
   oracle.farneback_np.pyramid_image on noise frames to float32 rounding."""
import numpy as np
import pytest

from oracle import farneback_np as fb

F32 = np.float32


def S(l):
    return 1 << l


def T(l):
    return 4 if l == 1 else 10 << (l - 2)


def NB(l):
    return 1 if l == 1 else 3 << (l - 2)


def K(l):
    return (T(l) + S(l) - 1) // S(l)


def reflect101(i, n):
    while i < 0 or i >= n:
        if n == 1:
            return 0
        i = -i if i < 0 else 2 * (n - 1) - i
    return i


def collapsed_filter(src, dst, scale):
    """base[d], weights[d][j] of the one-pass filter: c_j = (1 - a) k_j + a k_{j-1} at source index i0 - r + j."""
    sigma, ksz = fb.pyramid_blur_params(scale)
    k = fb.gaussian_kernel(ksz, sigma)
    i0, _, a = fb._resize_axis_coeffs(src, dst)
    r = ksz // 2
    w = np.zeros((dst, ksz + 1), dtype=F32)
    for j in range(ksz + 1):
        k0 = k[j] if j < ksz else F32(0)
        k1 = k[j - 1] if 1 <= j <= ksz else F32(0)
        w[:, j] = (F32(1) - a) * k0 + a * k1
    return i0 - r, w


@pytest.mark.parametrize('l', [1, 2, 3, 4, 5, 6])
@pytest.mark.parametrize('dst', [1, 2, 5, 34, 60])
def test_half_pyramid_constants_are_the_collapsed_filter(l, dst):
    src = dst << l
    base, w = collapsed_filter(src, dst, 0.5 ** l)
    assert w.shape[1] == T(l)
    assert np.array_equal(base, S(l) * np.arange(dst) - NB(l))
    assert np.all(w == w[0])                         # the same weights for every output sample
    assert K(l) <= 3 and T(l) <= K(l) * S(l)


def test_sizes_that_are_not_exact_decimations_are_not_uniform():
    # 1080 rows -> 68 (1080 / 16 = 67.5): the resize scale is 15.88, windows start 15 or 16 rows apart
    base, w = collapsed_filter(1080, 68, 0.5 ** 4)
    assert not np.array_equal(base, 16 * np.arange(68) - NB(4)) or not np.all(w == w[0])


def sweep_schedule(H, nlv, band_rows):
    """The loops of pyr_vsweep_kernel for one column: returns {level: {output row: [(tap, source row), ...]}} and the
    number of times each output was stored."""
    U = 1 << nlv
    h = {l: H >> l for l in range(1, nlv + 1)}
    taps = {l: {} for l in h}
    stored = {l: {} for l in h}
    h_top = h[nlv]
    for band in range((h_top + band_rows - 1) // band_rows):
        D0, D1 = band * band_rows, min((band + 1) * band_rows, h_top)
        acc = {l: [[] for _ in range(3)] for l in h}           # accumulators hold the (tap, row) products added so far
        for q in range(D0 - 1, D1 + 2):
            for i in range(U):
                row = reflect101(q * U + i, H)
                for l in h:
                    s, t, nb, k_live = S(l), T(l), NB(l), K(l)
                    ph = (i + nb) % s
                    for k in range(3):
                        if k < k_live and ph + k * s < t:
                            acc[l][k].append((ph + k * s, row))
                    if ph == s - 1:
                        dn = (U // s) * q + (i + nb) // s - (k_live - 1)
                        if D0 * (U // s) <= dn < min(D1 * (U // s), h[l]):
                            stored[l][dn] = stored[l].get(dn, 0) + 1
                            taps[l][dn] = list(acc[l][k_live - 1])
                        for k in range(2, 0, -1):
                            if k < k_live:
                                acc[l][k] = acc[l][k - 1]
                        acc[l][0] = []
    return taps, stored


@pytest.mark.parametrize('H,nlv,band_rows', [(32, 1, 16), (32, 2, 3), (64, 3, 8), (64, 3, 1), (48, 4, 2), (96, 3, 5),
                                              (16, 4, 1), (1080, 3, 34)])
def test_sweep_gives_every_output_its_taps_once_in_order(H, nlv, band_rows):
    assert H % (1 << nlv) == 0
    taps, stored = sweep_schedule(H, nlv, band_rows)
    for l in range(1, nlv + 1):
        hl = H >> l
        assert sorted(stored[l]) == list(range(hl)) and set(stored[l].values()) == {1}, (l, 'stored once each')
        for d in range(hl):
            want = [(j, reflect101(S(l) * d - NB(l) + j, H)) for j in range(T(l))]
            assert taps[l][d] == want, (l, d)


def _fma(a, b, c):
    # the exact product of two float32 fits in a float64; the float64 sum rounded to float32 differs from a true fma
    # only in rare double-rounding ties (the comparison below is tolerance-based)
    return (np.asarray(a, dtype=np.float64) * np.asarray(b, dtype=np.float64) + np.asarray(c, dtype=np.float64)).astype(F32)


def pyramid_by_kernels(img, nlv_v, levels):
    """The data path of the kernels: vertical sums per level (the sweep's accumulation order), level 1's horizontal
    pass from the thread's six columns (H1), 4-outputs-per-thread / one-output-per-thread horizontal passes above."""
    H, W = img.shape
    out = {}
    for l in range(1, levels + 1):
        hl, wl = H >> l, W >> l
        _, wy = collapsed_filter(H, hl, 0.5 ** l)
        _, wx = collapsed_filter(W, wl, 0.5 ** l)
        tmp = np.zeros((hl, W), dtype=F32)
        for d in range(hl):
            acc = np.zeros(W, dtype=F32)
            for j in range(T(l)):
                acc = _fma(wy[0, j], img[reflect101(S(l) * d - NB(l) + j, H)].astype(F32), acc)
            tmp[d] = acc
        res = np.zeros((hl, wl), dtype=F32)
        if l == 1:
            # thread = columns x .. x + 3 plus the reflected neighbours x - 1 and x + 4: outputs x / 2 and x / 2 + 1
            for x in range(0, W, 4):
                left = tmp[:, x - 1] if x >= 4 else tmp[:, x + 1]
                right = tmp[:, x + 4] if x + 4 < W else tmp[:, x + 2]
                c6 = [left, tmp[:, x], tmp[:, x + 1], tmp[:, x + 2], tmp[:, x + 3], right]
                o0 = np.zeros(hl, dtype=F32)
                o1 = np.zeros(hl, dtype=F32)
                for j in range(4):
                    o0 = _fma(wx[0, j], c6[j], o0)
                    o1 = _fma(wx[0, j], c6[2 + j], o1)
                res[:, x // 2], res[:, x // 2 + 1] = o0, o1
        else:
            off = (4 - NB(l) % 4) % 4
            for x in range(wl):
                a0 = S(l) * x - NB(l) - off                    # 16-byte group the window starts in
                assert a0 % 4 == 0
                acc = np.zeros(hl, dtype=F32)
                for j in range(T(l)):
                    acc = _fma(wx[0, j], tmp[:, reflect101(a0 + off + j, W)], acc)
                res[:, x] = acc
        out[l] = res
    return out


@pytest.mark.parametrize('size,levels', [((64, 48), 3), ((96, 64), 3), ((256, 128), 5), ((128, 64), 6)])
def test_restated_kernels_match_the_oracle_pyramid(size, levels):
    W, H = size
    rng = np.random.default_rng(W * H)
    img = rng.integers(0, 256, size=(H, W), dtype=np.uint8)
    got = pyramid_by_kernels(img, levels, levels)
    for l in range(1, levels + 1):
        ref = fb.pyramid_image(img, 0.5 ** l, W >> l, H >> l)
        assert np.abs(got[l] - ref).max() < 5e-4, (l, float(np.abs(got[l] - ref).max()))      # 0..255 scale
