"""The tcgen05 int8 Ozaki kernels (stheno.jl_b200/csrc/ozaki.cu) bit for bit against their exact model.

The kernels' arithmetic is deterministic: the seven digit-group accumulators are exact int32 sums, the epilogue
adds them into fp64 in a fixed order and applies one fma (SYRK / plain) or one product (STORE) with the power-of-two
row scales.  oracle/device_algorithms.py restates that order (oz_groups, oz_epilogue_acc, oz_update, oz_store), so
every output here -- digit planes, row scales, int32 accumulators, the packed matrix after a trailing update, dense
products and the panel solve -- must be EQUAL to the model, compared on the float64 bit patterns.  A group read
before its last MMA landed, an accumulator released too early or a stale phase bit changes low bits that the
end-to-end tolerances of tests/test_gpu_parity.py cannot see.

The kernels are driven through build/liboz_hooks.so (tests/csrc/oz_hooks.cu): host buffers in, one launch of the
shipped launcher, host buffers out."""
import ctypes as C
import functools
import math
import os

import numpy as np
import pytest

from oracle import device_algorithms as da

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOOKS_PATH = os.path.join(ROOT, "build", "liboz_hooks.so")
NB, S, KMAX = 128, 7, 512
MODES = [0, 1, 2, 4, 6, 8, 10, 12, 16]     # every kernel instance OZ_DISPATCH / the ring kernel can launch
BIAS = 0x808080808080


# ---------------------------------------------------------------------------------------------------------
# hooks
# ---------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def hooks(sb):
    sb.lib.load()            # RTLD_GLOBAL: provides the launchers the hooks call
    if not os.path.exists(HOOKS_PATH):
        pytest.fail(f"{HOOKS_PATH} not built: run stheno.jl_b200/csrc/build.sh")
    h = C.CDLL(HOOKS_PATH)
    vp, i32, i64 = C.c_void_p, C.c_int, C.c_int64
    h.oz_hooks_last_error.restype = C.c_char_p
    h.oz_hooks_sm_count.argtypes = [C.POINTER(i32)]
    h.oz_hooks_slice.argtypes = [vp, i64, i32, vp, vp, vp, i64, i64, i64, i64, vp, vp, vp]
    h.oz_hooks_syrk_packed.argtypes = [vp, i64, vp, vp, i64, i32, i64, i64, i32, i32, i32, i32, i64, i64, vp]
    h.oz_hooks_gemm_plain.argtypes = [vp, i64, i64, i64, i32, vp, vp, i64, i64, vp, vp, i64, i64, i32]
    h.oz_hooks_panel_solve.argtypes = [C.POINTER(vp), vp, i64, vp, vp, i64, i64, vp, vp]
    return h


def _ok(h, rc):
    assert rc == 0, f"hook failed ({rc}): {h.oz_hooks_last_error().decode()}"


def _p(a):
    assert a.flags.c_contiguous
    return a.ctypes.data


def _sm_count(h):
    n = C.c_int(0)
    _ok(h, h.oz_hooks_sm_count(C.byref(n)))
    return n.value


def assert_bits_equal(got, want, what):
    g, w = np.ascontiguousarray(got), np.ascontiguousarray(want)
    assert g.shape == w.shape and g.dtype == w.dtype
    gi = g.view(np.int64) if g.dtype == np.float64 else g
    wi = w.view(np.int64) if w.dtype == np.float64 else w
    bad = np.argwhere(gi != wi)
    if len(bad):
        i = tuple(bad[0])
        raise AssertionError(f"{what}: {len(bad)} of {g.size} entries differ; first at {i}: got {g[i]!r}, want {w[i]!r}")


def _planes(digits, rng):
    """[7][rows][512] plane buffer holding digits[:, :, :K]; the bytes past K are garbage the kernels must not read"""
    _, rows, K = digits.shape
    out = rng.integers(-128, 128, (S, rows, KMAX), dtype=np.int8)
    out[:, :, :K] = digits
    return np.ascontiguousarray(out)


def _rows(rng, m, K, spread=8.0):
    """rows of very different magnitudes, some exact zeros and a few all-zero rows"""
    P = rng.standard_normal((m, K)) * np.exp(rng.uniform(-spread, spread, (m, 1)))
    P[rng.random((m, K)) < 0.02] = 0.0
    P[rng.random(m) < 0.01] = 0.0
    return P


# ---------------------------------------------------------------------------------------------------------
# slicer
# ---------------------------------------------------------------------------------------------------------
def _special_rows(K, rng):
    """128 rows x K values that probe the slicer's edges; the largest entry sits at varying columns, also in the
    last 128-column segment (the row max is reduced across segments)"""
    R = np.zeros((NB, K))
    i = 0

    def put(row_vals, big):
        nonlocal i
        R[i] = row_vals
        R[i, (37 * i + 11) % K] = big
        i += 1

    small = lambda scale: rng.uniform(-scale, scale, K) * 0.4
    i += 1                                                          # row 0: all zero
    for k in (3, -7, 40):
        put(small(2.0 ** k), 2.0 ** k)                              # max exactly 2^k
        put(small(2.0 ** k), np.nextafter(2.0 ** k, 0.0))           # 2^k - ulp: one ilogb lower
        put(small(2.0 ** k), -(2.0 ** k))                           # negative maxima
        put(small(2.0 ** k), -np.nextafter(2.0 ** k, 0.0))
    for t in (1e-280, 1e280):                                       # the range the slicer accepts: (1e-280, 1e280)
        for v in (np.nextafter(t, 0.0), t, np.nextafter(t, np.inf)):
            put(small(v) * 0.5, v)
            put(small(v) * 0.5, -v)
    sub = np.full(K, 0.0)
    sub[::3], sub[1::3] = 5e-324, -2.5e-310                         # subnormal entries inside normal rows
    put(sub * 1.0, 3.0)
    put(sub * 1.0, np.nextafter(1e-280, 1.0) * 7)
    # rint ties: x 2^(55 - e) = n + 1/2 exactly (round half to even), e = 1 from the max 0.75
    n = np.concatenate([np.arange(-40, 40), rng.integers(-2 ** 52, 2 ** 52, 40)]).astype(np.float64)
    ties = (n + 0.5) * 2.0 ** (1 - 55)
    for c0 in range(0, len(ties), K - 1):
        v = np.zeros(K)
        chunk = ties[c0:c0 + K - 1]
        v[:len(chunk)] = chunk
        R[i] = v
        R[i, K - 1] = 0.75
        i += 1
    # biased bytes that carry through every digit
    Zs = [-1, 1, -2 ** 48, 2 ** 48 - 1, 0x7F7F7F7F7F80, 0x7F7F7F7F7F7F, -BIAS, -BIAS - 1, -BIAS + 1,
          0xFFFFFFFFFF, -0xFFFFFFFFFF, 2 ** 53 - 2, -(2 ** 53 - 2)]
    v = np.zeros(K)
    v[:len(Zs)] = np.ldexp(np.array(Zs, dtype=np.float64), 1 - 55)
    v[-1] = 0.75
    R[i] = v
    i += 1
    R[i:] = _rows(rng, NB - i, K, 20.0)
    return R


def _gather(src, nseg, off, ld, rbs, rb, r):
    """row r of row block rb of the source panel: K = 128 nseg values"""
    return np.concatenate([src[off[q] + rb * rbs[q] + np.arange(NB) * ld[q] + r] for q in range(nseg)])


@pytest.mark.parametrize("layout", ["tiled", "plain"])
@pytest.mark.parametrize("nseg", [1, 2, 3, 4])
def test_slicer_equals_model(hooks, layout, nseg):
    rng = np.random.default_rng(100 + nseg + (layout == "tiled") * 10)
    K = NB * nseg
    nrb, rb_lo, out_row_base = 3, 1, 256          # source row blocks 1..3 -> plane rows 384 .. 767
    plane_rows = out_row_base + (rb_lo + nrb) * NB + NB
    total_rb = rb_lo + nrb
    rows = np.concatenate([_special_rows(K, rng), _rows(rng, (total_rb - 1) * NB, K, 30.0)])   # [rb][r] -> row
    if layout == "tiled":
        ld, rbs = [NB + 4] * nseg, [NB * (NB + 4)] * nseg
        seg_elems = total_rb * NB * (NB + 4)
    else:
        height = total_rb * NB + 40                     # column-major panels with their own leading dimensions
        ld = [height + 8 * q for q in range(nseg)]
        rbs = [NB] * nseg
        seg_elems = None
    sizes = [seg_elems if seg_elems else ld[q] * NB for q in range(nseg)]
    off = list(np.cumsum([0] + sizes[:-1]) + 5)        # segments packed into one buffer, not aligned to each other
    src = rng.standard_normal(int(off[-1] + sizes[-1] + 5)) * 1e300   # padding rows / gaps: must not be read
    # the special rows go into the first source row block that is sliced (rb_lo)
    perm = np.concatenate([np.arange(NB, rb_lo * NB + NB), np.arange(NB), np.arange(rb_lo * NB + NB, total_rb * NB)])
    rows = rows[perm]
    for rb in range(total_rb):
        for q in range(nseg):
            blk = rows[rb * NB:(rb + 1) * NB, q * NB:(q + 1) * NB]           # [r][k]
            idx = off[q] + rb * rbs[q] + np.arange(NB)[None, :] * ld[q] + np.arange(NB)[:, None]
            src[idx] = blk
    planes = rng.integers(-128, 128, (S, plane_rows, KMAX), dtype=np.int8)
    scale = rng.standard_normal(plane_rows)
    expo = rng.integers(-1000, 1000, plane_rows).astype(np.int32)
    want_p, want_s, want_e = planes.copy(), scale.copy(), expo.copy()
    P = rows[rb_lo * NB:total_rb * NB]
    assert np.array_equal(_gather(src, nseg, off, ld, rbs, rb_lo, 5), P[5])
    d, s = da.oz_slice(P)
    pr = slice(out_row_base + rb_lo * NB, out_row_base + total_rb * NB)
    want_p[:, pr, :K] = d
    want_s[pr] = s
    want_e[pr] = da.oz_row_exponents(P)
    offs, lds, rbss = (np.array(a, dtype=np.int64) for a in (off, ld, rbs))
    _ok(hooks, hooks.oz_hooks_slice(_p(src), src.size, nseg, _p(offs), _p(lds), _p(rbss), rb_lo, nrb, out_row_base,
                                    plane_rows, _p(planes), _p(scale), _p(expo)))
    assert_bits_equal(expo, want_e, "exponents")
    assert_bits_equal(scale, want_s, "scales")
    assert_bits_equal(planes, want_p, "digit planes")
    assert (want_e[pr] == da.OZ_NO_EXPO).sum() >= 4 and (want_p[1:, pr, :K] == -128).any()


# ---------------------------------------------------------------------------------------------------------
# packed SYRK
# ---------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _syrk_problem(Np):
    rng = np.random.default_rng(Np)
    d, s = da.oz_slice(_rows(rng, Np, KMAX))
    return rng.standard_normal(da.packed_size(Np)), _planes(d, rng), s, d


@functools.lru_cache(maxsize=None)
def _syrk_model(Np, nseg):
    C0, _, s, d = _syrk_problem(Np)
    return da.oz_syrk_update(C0, Np, d[:, :, :NB * nseg], s)


def _syrk(h, Np, nseg=4, k=0, jlo=0, jhi=None, rank=0, world=1, mode=8, reserve=0, tile_lo=0, tile_hi=0, C=None,
          dbg=False):
    C0, planes, s, _ = _syrk_problem(Np)
    out = (C0 if C is None else C).copy()
    g = np.full((S, NB, 64), -7, dtype=np.int32) if dbg else None
    _ok(h, h.oz_hooks_syrk_packed(_p(out), Np, _p(planes), _p(s), k, nseg, jlo, Np // NB if jhi is None else jhi,
                                  rank, world, mode, reserve, tile_lo, tile_hi, _p(g) if dbg else None))
    return (out, g) if dbg else out


def _syrk_want(Np, nseg, tiles, C=None):
    C0 = _syrk_problem(Np)[0]
    return da.oz_apply_tiles(C0 if C is None else C, _syrk_model(Np, nseg), Np, tiles)


@pytest.mark.parametrize("mode", MODES)
def test_syrk_every_instance(hooks, mode):
    """Np = 2048, K = 512, trailing update of step k = 1: the whole packed matrix, and the raw int32 accumulators
    of tile 0 (block (2, 2), left half)."""
    Np, k = 2048, 1
    got, g = _syrk(hooks, Np, k=k, mode=mode, dbg=True)
    assert_bits_equal(got, _syrk_want(Np, 4, da.oz_syrk_tiles(Np // NB, k, 0, Np // NB)), f"packed matrix, mode {mode}")
    d = _syrk_problem(Np)[3]
    r0 = (k + 1) * NB
    G = da.oz_groups(d[:, r0:r0 + NB], d[:, r0:r0 + 64])
    assert_bits_equal(g, np.stack(G).astype(np.int32), f"tile-0 accumulators, mode {mode}")


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("nseg", [1, 2, 3])
def test_syrk_short_k(hooks, nseg, mode):
    Np = 1024
    got = _syrk(hooks, Np, nseg=nseg, k=0, mode=mode)
    assert_bits_equal(got, _syrk_want(Np, nseg, da.oz_syrk_tiles(Np // NB, 0, 0, Np // NB)), "packed matrix")


@pytest.mark.parametrize("mode", [8, 16])
@pytest.mark.parametrize("k,jlo,jhi", [(0, 3, 7), (2, 0, 5), (4, 9, 10), (0, 15, 16), (6, 0, 99)])
def test_syrk_column_ranges(hooks, k, jlo, jhi, mode):
    Np = 2048
    got = _syrk(hooks, Np, k=k, jlo=jlo, jhi=jhi, mode=mode)
    assert_bits_equal(got, _syrk_want(Np, 4, da.oz_syrk_tiles(Np // NB, k, jlo, jhi)), "packed matrix")


@pytest.mark.parametrize("mode", [8, 16])
@pytest.mark.parametrize("world", [1, 2, 3])
def test_syrk_rank_ownership(hooks, world, mode):
    """Each rank updates only its block columns; all ranks applied in turn give the whole update."""
    Np, k, nblk = 2048, 1, 16
    C = _syrk_problem(Np)[0]
    for rank in range(world):
        got = _syrk(hooks, Np, k=k, rank=rank, world=world, mode=mode, C=C)
        assert_bits_equal(got, _syrk_want(Np, 4, da.oz_syrk_tiles(nblk, k, 0, nblk, rank, world), C=C),
                          f"rank {rank} of {world}")
        C = got
    assert_bits_equal(C, _syrk_want(Np, 4, da.oz_syrk_tiles(nblk, k, 0, nblk)), "all ranks")


@pytest.mark.parametrize("mode", [8, 16, 2])
def test_syrk_tile_range_split(hooks, mode):
    """cholesky_wide's T^B: part 1 on a persistent grid that leaves SMs free, part 2 on the whole GPU."""
    Np, k, jlo = 2048, 0, 5
    nblk = Np // NB
    total = len(da.oz_syrk_tiles(nblk, k, jlo, nblk))
    n1 = 97
    part1 = _syrk(hooks, Np, k=k, jlo=jlo, mode=mode, reserve=8, tile_lo=0, tile_hi=n1)
    assert_bits_equal(part1, _syrk_want(Np, 4, da.oz_syrk_tiles(nblk, k, jlo, nblk, tile_hi=n1)), "part 1")
    both = _syrk(hooks, Np, k=k, jlo=jlo, mode=mode, tile_lo=n1, tile_hi=total, C=part1)
    assert_bits_equal(both, _syrk_want(Np, 4, da.oz_syrk_tiles(nblk, k, jlo, nblk)), "parts 1 + 2")


@pytest.mark.parametrize("mode", [8, 16, 0, 12])
@pytest.mark.parametrize("reserve", ["0", "sms-2", "-1", "-3"])
def test_syrk_grid_shapes(hooks, reserve, mode):
    """Persistent grids (many tiles per CTA when all but two SMs are left free: the TMEM phase bits flip dozens
    of times) and chunked CTAs of 1 / 3 tiles."""
    Np, k = 2048, 0
    r = _sm_count(hooks) - 2 if reserve == "sms-2" else int(reserve)
    got = _syrk(hooks, Np, k=k, mode=mode, reserve=r)
    assert_bits_equal(got, _syrk_want(Np, 4, da.oz_syrk_tiles(Np // NB, k, 0, Np // NB)), f"reserve_sms {r}")


def test_syrk_large(hooks):
    Np, k = 4096, 2
    got = _syrk(hooks, Np, k=k, mode=8)
    assert_bits_equal(got, _syrk_want(Np, 4, da.oz_syrk_tiles(Np // NB, k, 0, Np // NB)), "packed matrix")


@pytest.mark.parametrize("mode", [8, 16])
def test_int32_headroom_and_signed_digits(hooks, mode):
    """Rows whose six low digits are all -128 and whose top digit is at its extreme (64 or -63): the accumulators of
    tile 0 must equal the model's integers (signed kind::i8 at -128, no int32 wrap) and the matrix the model."""
    Np, K = 1024, KMAX
    rng = np.random.default_rng(77)
    P = _rows(rng, Np, K)
    for i in range(NB, 3 * NB):                         # block rows 1 and 2: tile 0 of k = 0 is block (1, 1)
        d0 = 64 if (i // 3) % 2 == 0 else -63
        P[i] = math.ldexp(float(d0 * 2 ** 48 - BIAS), int(rng.integers(-20, 20)) - 55)
    d, s = da.oz_slice(P)
    assert np.all(d[1:, NB:3 * NB] == -128) and set(np.unique(d[0, NB:3 * NB])) == {64, -63}
    planes = _planes(d, rng)
    C0 = rng.standard_normal(da.packed_size(Np))
    out, g = C0.copy(), np.zeros((S, NB, 64), dtype=np.int32)
    _ok(hooks, hooks.oz_hooks_syrk_packed(_p(out), Np, _p(planes), _p(s), 0, 4, 0, Np // NB, 0, 1, mode, 0, 0, 0,
                                          _p(g)))
    G = np.stack(da.oz_groups(d[:, NB:2 * NB], d[:, NB:NB + 64]))
    assert np.abs(G).max() >= 2 ** 25
    assert_bits_equal(g, G.astype(np.int32), "tile-0 accumulators")
    want = da.oz_apply_tiles(C0, da.oz_syrk_update(C0, Np, d, s), Np, da.oz_syrk_tiles(Np // NB, 0, 0, Np // NB))
    assert_bits_equal(out, want, "packed matrix")


# ---------------------------------------------------------------------------------------------------------
# plain mode: C[M x Ncols] -= A B^T
# ---------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _plain_sets():
    rng = np.random.default_rng(5)
    dA, sA = da.oz_slice(_rows(rng, 1024, KMAX, 6.0))
    dB, sB = da.oz_slice(_rows(rng, 768, KMAX, 3.0) * 1e-3)
    return (_planes(dA, rng), sA, dA), (_planes(dB, rng), sB, dB)


def _plain(h, M, Ncols, nseg, mode, rowA0=384, rowB0=192):
    (pA, sA, dA), (pB, sB, dB) = _plain_sets()
    rng = np.random.default_rng(M + Ncols + nseg)
    ldc = M + 40
    Cm = np.ascontiguousarray(rng.standard_normal((Ncols, ldc)))      # column-major ldc x Ncols
    want = Cm.copy()
    K = NB * nseg
    acc = da.oz_epilogue_acc(da.oz_groups(dA[:, rowA0:rowA0 + M, :K], dB[:, rowB0:rowB0 + Ncols, :K]))
    want[:, :M] = da.oz_update(Cm[:, :M].T, sA[rowA0:rowA0 + M], sB[rowB0:rowB0 + Ncols], acc).T
    _ok(h, h.oz_hooks_gemm_plain(_p(Cm), ldc, M, Ncols, nseg, _p(pA), _p(sA), pA.shape[1], rowA0, _p(pB), _p(sB),
                                 pB.shape[1], rowB0, mode))
    assert_bits_equal(Cm, want, f"C, M {M} Ncols {Ncols} nseg {nseg} mode {mode}")


@pytest.mark.parametrize("nseg", [1, 2, 3, 4])
@pytest.mark.parametrize("M,Ncols", [(128, 128), (128, 512), (384, 128), (384, 512)])
def test_plain_product(hooks, M, Ncols, nseg):
    _plain(hooks, M, Ncols, nseg, 8)


@pytest.mark.parametrize("mode", MODES)
def test_plain_product_every_instance(hooks, mode):
    _plain(hooks, 384, 512, 3, mode, rowA0=128, rowB0=64)


# ---------------------------------------------------------------------------------------------------------
# STORE mode: the panel solve X = A inv(L_512)^T
# ---------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _inv_l512():
    rng = np.random.default_rng(11)
    G = rng.standard_normal((512, 520))
    _, W = da.wide_panel_factor(G @ G.T / 520 + 0.3 * np.eye(512))
    return W


@pytest.mark.parametrize("M,garbage", [(128, False), (640, False), (1280, False), (640, True)])
def test_panel_solve(hooks, M, garbage):
    """X equals the model over all four block columns (each with its own leading dimension; rows past M untouched).
    With garbage in the strictly upper 128-blocks of W the result must not change: block column q of X only reads
    K < 128 (q + 1)."""
    rng = np.random.default_rng(M + garbage)
    W = _inv_l512()
    blk = np.repeat(np.arange(4), NB)
    upper = blk[:, None] < blk[None, :]             # the strictly upper 128-blocks
    assert np.all(W[upper] == 0)
    dW, sW = da.oz_slice(W)
    Wg = W.copy()
    if garbage:
        rmax = np.max(np.abs(W), axis=1, keepdims=True)
        Wg[upper] = (rng.uniform(-0.9, 0.9, W.shape) * rmax)[upper]      # below each row's max: same exponents
    dWg, sWg = da.oz_slice(Wg)
    assert np.array_equal(sWg, sW) and (not garbage or (dWg != dW).any())
    rowA0, rowsA = 256, 256 + M + 128
    A = _rows(rng, rowsA, KMAX, 4.0)
    dA, sA = da.oz_slice(A)
    pA, pW = _planes(dA, rng), _planes(dWg, rng)
    ldx = np.array([M + 384, M + 256, M + 128, M], dtype=np.int64)
    X = [np.ascontiguousarray(rng.standard_normal((NB, ld))) for ld in ldx]    # column-major ld x 128
    want = [x.copy() for x in X]
    for q in range(4):
        K = NB * (q + 1)
        acc = da.oz_epilogue_acc(da.oz_groups(dA[:, rowA0:rowA0 + M, :K], dW[:, q * NB:(q + 1) * NB, :K]))
        want[q][:, :M] = da.oz_store(sA[rowA0:rowA0 + M], sW[q * NB:(q + 1) * NB], acc).T
    ptrs = (C.c_void_p * 4)(*[_p(x) for x in X])
    _ok(hooks, hooks.oz_hooks_panel_solve(ptrs, _p(ldx), M, _p(pA), _p(sA), rowsA, rowA0, _p(pW), _p(sW)))
    for q in range(4):
        assert_bits_equal(X[q], want[q], f"X block column {q}")
