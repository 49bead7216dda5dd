"""CPU pins for the numerical schemes the CUDA library uses in place of LAPACK's dpotrf / dtrsm (the reference's
`cholesky(Symmetric(cov(fx)))`, SURVEY.md App. A): the int8 digit-plane product, the wide panel phase and the
peer-to-peer exchange protocol -- restated in NumPy in oracle/device_algorithms.py and checked here against
exact integer arithmetic, LAPACK and randomised interleavings.  The device kernels are compared with the same
quantities on the GPU: tests/test_gpu_ozaki_exact.py demands bit-for-bit equality of every tcgen05 kernel instance
with the exact model pinned here; tests/test_gpu_parity.py compares the whole pipeline with the oracle."""
import math
from fractions import Fraction

import numpy as np
import pytest

from oracle import device_algorithms as da


def _rows(rng, m, K, spread):
    """rows with very different magnitudes and a few exact zeros"""
    P = rng.standard_normal((m, K)) * np.exp(rng.uniform(-spread, spread, (m, 1)))
    P[rng.random((m, K)) < 0.02] = 0.0
    return P


def test_digit_planes_reconstruct_to_56_bits():
    rng = np.random.default_rng(1)
    P = _rows(rng, 64, 96, 30.0)
    P[5] = 0.0                                     # an all-zero row has scale 0 and zero digits
    d, s = da.oz_slice(P)
    assert d.dtype == np.int8 and d.shape == (7, 64, 96)
    R = da.oz_reconstruct(d, s)
    mx = np.max(np.abs(P), axis=1, keepdims=True)
    assert np.all(np.abs(R - P) <= mx * 2.0 ** -53)  # half an ulp of the 56-bit grid is 2^-56 * 2^(e) <= mx 2^-54
    assert s[5] == 0.0 and not d[:, 5].any()
    # balanced digits: the six low planes really use the signed range
    assert d[1:].min() == -128 and d[1:].max() == 127


def test_digit_planes_are_an_exact_integer_identity():
    """Z = sum_p d_p 256^(6-p) holds exactly (checked with Python integers), including negative values and carries."""
    rng = np.random.default_rng(2)
    P = _rows(rng, 8, 40, 5.0)
    d, s = da.oz_slice(P)
    e = np.round(np.log2(s)).astype(int) + 31
    for i in range(P.shape[0]):
        for k in range(P.shape[1]):
            Z = int(np.rint(np.ldexp(P[i, k], 55 - e[i])))
            assert Z == sum(int(d[p, i, k]) * 256 ** (6 - p) for p in range(7))


def test_digit_plane_product_matches_exact_arithmetic():
    rng = np.random.default_rng(3)
    m, n, K = 24, 16, 512
    A, B = _rows(rng, m, K, 8.0), _rows(rng, n, K, 8.0)
    dA, sA = da.oz_slice(A)
    dB, sB = da.oz_slice(B)
    C, gmax = da.oz_product(dA, sA, dB, sB)
    assert gmax < 2 ** 31                           # int32 accumulators: 7 pairs x 512 x 2^14 < 2^31
    assert 7 * K * 128 * 128 < 2 ** 31
    exact = np.array([[float(sum(Fraction(a) * Fraction(b) for a, b in zip(A[i], B[j]))) for j in range(n)] for i in range(m)])
    bound = np.max(np.abs(A), axis=1)[:, None] * np.max(np.abs(B), axis=1)[None, :]
    err = np.abs(C - exact) / bound
    # dropped pairs (p + q > 6) + 56-bit rounding: a few 1e-15 of max|row_i| max|row_j| per unit of sqrt(K)
    assert err.max() < 2e-13, err.max()
    # and it is not worse than plain fp64 accumulation by more than that
    assert np.abs(A @ B.T - exact).max() / bound.max() < 1e-13


def test_dropping_low_digit_pairs_is_what_limits_the_accuracy():
    rng = np.random.default_rng(4)
    A, B = rng.standard_normal((8, 256)), rng.standard_normal((8, 256))
    dA, sA = da.oz_slice(A)
    dB, sB = da.oz_slice(B)
    full, _ = da.oz_product(dA, sA, dB, sB, max_group=12)     # all 49 pairs: exact up to the 56-bit rounding
    kept, _ = da.oz_product(dA, sA, dB, sB)                   # the kernel's 28 pairs
    exact = np.array([[float(sum(Fraction(a) * Fraction(b) for a, b in zip(A[i], B[j]))) for j in range(8)] for i in range(8)])
    assert np.abs(full - exact).max() < 1e-14
    assert np.abs(kept - exact).max() < 5e-13
    assert np.abs(kept - exact).max() >= np.abs(full - exact).max()


@pytest.mark.parametrize("m_below", [0, 128, 640])
def test_wide_panel_phase_equals_lapack(m_below):
    rng = np.random.default_rng(5)
    w, n = 512, 512 + m_below
    G = rng.standard_normal((n, n + 8))
    S = G @ G.T / n + 0.5 * np.eye(n)
    L = np.linalg.cholesky(S)
    out, W = da.wide_panel_factor(S[:, :w].copy())
    np.testing.assert_allclose(np.tril(out[:w]), L[:w, :w], rtol=0, atol=2e-13)
    np.testing.assert_allclose(out[w:], L[w:, :w], rtol=0, atol=2e-13)
    # the identity rows hold inv(L_512): block lower triangular, and W L = I
    np.testing.assert_allclose(W @ L[:w, :w], np.eye(w), atol=1e-12)
    assert np.all(W[:128, 128:] == 0.0) and np.all(W[128:256, 256:] == 0.0)


def test_wide_panel_phase_with_the_digit_plane_product():
    """the device's panel solve: X = A inv(L_512)^T through int8 digit planes of both operands"""
    rng = np.random.default_rng(6)
    w, n = 512, 512 + 256
    G = rng.standard_normal((n, n + 8))
    S = G @ G.T / n + 0.1 * np.eye(n)
    d = np.exp(rng.uniform(-4, 4, n))
    S = S * d[:, None] * d[None, :]                 # badly scaled rows / columns, still SPD
    L = np.linalg.cholesky(S)

    def product(A, Wm):
        dA, sA = da.oz_slice(A)
        dW, sW = da.oz_slice(Wm)
        return da.oz_product(dA, sA, dW, sW)[0]

    out, _ = da.wide_panel_factor(S[:, :w].copy(), product=product)
    scale = np.sqrt(np.diag(S))[w:, None]           # |L_ij| <= sqrt(S_ii): the natural error unit of a Cholesky row
    assert np.max(np.abs(out[w:] - L[w:, :w]) / scale) < 1e-11


@pytest.mark.parametrize("world", [2, 3, 4, 5, 8])
def test_p2p_exchange_protocol_is_safe_and_live(world):
    rng = np.random.default_rng(100 + world)
    for trial in range(30):
        ncols = int(rng.integers(5, 90))
        base = [int(b) for b in rng.integers(0, 50, world)] if trial % 2 else None   # counters survive across factorisations
        mdl = da.P2PExchangeModel(world, ncols, slots=8, base=base)
        bias = None if trial % 3 else [1e-3 if r == trial % world else 1.0 for r in range(world)]   # one very slow rank
        mdl.run(rng, bias)
        for r in range(world):
            assert sorted(mdl.got[r]) == [k for k in range(ncols) if k % world != r]


def test_p2p_exchange_without_the_slot_guard_is_caught():
    """Sanity of the model, and why the guard exists: with 8 ranks only half of them own a column in a given
    outer step, so a slow rank is not implicitly waited for; without the ack guard a fast owner overwrites the
    slot the slow rank still has to pull."""
    rng = np.random.default_rng(7)
    hit = 0
    for trial in range(40):
        mdl = da.P2PExchangeModel(8, 64, slots=8, guard=False)
        try:
            mdl.run(rng, [1e-3 if r == trial % 8 else 1.0 for r in range(8)])
        except AssertionError as e:
            assert "overwrites slot" in str(e) or "expected column" in str(e)
            hit += 1
    assert hit > 0


def test_blas_groups_equal_the_int64_accumulators():
    """oz_groups (float64 BLAS on the int8 digits) is exact: it equals the int64 sums of oz_product's loop."""
    rng = np.random.default_rng(8)
    dA, _ = da.oz_slice(_rows(rng, 40, 512, 10.0))
    dB, _ = da.oz_slice(_rows(rng, 24, 512, 10.0))
    dA[1:, :3] = -128                               # extreme digits in a few columns
    dB[1:, :3] = -128
    G = da.oz_groups(dA, dB)
    for g in range(7):
        ref = sum(dA[p].astype(np.int64) @ dB[g - p].astype(np.int64).T for p in range(g + 1))
        assert np.array_equal(G[g].astype(np.int64), ref) and np.array_equal(G[g], ref.astype(np.float64))


def test_epilogue_model_agrees_with_the_digit_plane_product():
    """The epilogue-ordered model (groups -> weighted fp64 sum -> (s_i s_j) acc) is oz_product bit for bit on rows
    of normal magnitude, and the SYRK update is C - that product rounded once."""
    rng = np.random.default_rng(9)
    A, B = _rows(rng, 32, 384, 6.0), _rows(rng, 20, 384, 6.0)
    A[3] = 0.0
    dA, sA = da.oz_slice(A)
    dB, sB = da.oz_slice(B)
    acc = da.oz_epilogue_acc(da.oz_groups(dA, dB))
    X = da.oz_store(sA, sB, acc)
    assert np.array_equal(X.view(np.int64), da.oz_product(dA, sA, dB, sB)[0].view(np.int64))
    C = rng.standard_normal((32, 20))
    assert np.array_equal(da.oz_update(C, sA, sB, acc), C - X)


def test_slicer_exponents_at_the_ilogb_and_range_boundaries():
    P = np.zeros((6, 4))
    P[0, 1] = 8.0                                   # max exactly 2^3: e = 3 + 2
    P[1, 2] = np.nextafter(8.0, 0.0)                # 2^3 - ulp: e = 2 + 2
    P[2, 0] = -8.0                                  # negative maximum
    P[3, 3] = 1e-280                                # not above 1e-280: zero row
    P[4, 3] = np.nextafter(1e-280, 1.0)
    P[5, 0] = np.nextafter(1e280, 0.0)
    e = da.oz_row_exponents(P)
    assert list(e[:3]) == [5, 4, 5] and e[3] == da.OZ_NO_EXPO
    assert e[4] == int(np.frexp(1e-280)[1]) + 1 and e[5] == int(np.frexp(1e280)[1]) + 1


def test_headroom_rows_give_extreme_digits():
    """Z = 64 2^48 - 0x808080808080 slices to d_0 = 64 and six digits -128 (the largest digits a row can have);
    Z = -63 2^48 - 0x808080808080 to d_0 = -63 and six digits -128."""
    bias = 0x808080808080
    for d0 in (64, -63):
        Z = d0 * 2 ** 48 - bias
        x = np.full((1, 8), math.ldexp(float(Z), 1 - 55))          # e = 1
        d, s = da.oz_slice(x)
        assert s[0] == 2.0 ** -30 and np.all(d[0] == d0) and np.all(d[1:] == -128)


def test_syrk_tile_set_follows_the_launcher():
    nblk = 12
    for k, jlo, jhi in [(0, 0, nblk), (2, 0, 7), (0, 5, 6), (3, 9, 30)]:
        full = da.oz_syrk_tiles(nblk, k, jlo, jhi)
        lo, hi = max(jlo, k + 1), min(jhi, nblk)
        assert len(full) == 2 * sum(nblk - J for J in range(lo, hi))
        assert full == sorted(full, key=lambda t: (t[1], t[0], t[2]))
        for world in (2, 3):
            parts = [da.oz_syrk_tiles(nblk, k, jlo, jhi, r, world) for r in range(world)]
            assert sorted(sum(parts, [])) == sorted(full)
            assert all(J % world == r for r, part in enumerate(parts) for _, J, _ in part)
        n1 = len(full) // 3
        assert da.oz_syrk_tiles(nblk, k, jlo, jhi, tile_hi=n1) + da.oz_syrk_tiles(nblk, k, jlo, jhi, tile_lo=n1) == full


def test_packed_layout_helpers():
    Np = 512
    buf = np.arange(da.packed_size(Np), dtype=np.float64)
    assert da.packed_size(Np) == Np * (Np + 128) // 2
    for J in range(Np // 128):
        V = da.packed_column(buf, Np, J)
        ld = Np - 128 * J
        assert V.shape == (ld, 128)
        assert V[5, 7] == da.packed_offset(Np, J) + 7 * ld + 5


def test_syrk_model_is_the_lower_triangle_of_the_dense_update():
    rng = np.random.default_rng(10)
    Np, K = 384, 256
    P = _rows(rng, Np, K, 4.0)
    d, s = da.oz_slice(P)
    C = rng.standard_normal(da.packed_size(Np))
    new = da.oz_syrk_update(C, Np, d, s)
    dense = da.oz_store(s, s, da.oz_epilogue_acc(da.oz_groups(d, d)))
    for J in range(3):
        r0 = 128 * J
        want = da.packed_column(C, Np, J) - dense[r0:, r0:r0 + 128]
        assert np.array_equal(da.packed_column(new, Np, J), want)
    half = da.oz_syrk_tiles(3, 0, 0, 3, tile_hi=3)            # (1, 1, 0), (1, 1, 1), (2, 1, 0)
    part = da.oz_apply_tiles(C, new, Np, half)
    V, Vn = da.packed_column(part, Np, 1), da.packed_column(new, Np, 1)
    assert np.array_equal(V[:, :64], Vn[:, :64]) and np.array_equal(V[:128, 64:], Vn[:128, 64:])
    assert np.array_equal(V[128:, 64:], da.packed_column(C, Np, 1)[128:, 64:])
    assert np.array_equal(da.packed_column(part, Np, 0), da.packed_column(C, Np, 0))
