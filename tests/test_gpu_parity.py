"""GPU parity: the CUDA path (through the C ABI) against the CPU oracle on identical inputs.

Tolerances: fp64, rtol 1e-10 on logpdf / posterior (BASELINE.json north_star); covariance
entries to 1e-13 absolute (1-D inputs follow the reference's rounding sequence exactly, so they
are in practice bit-identical up to the ulp of exp()).
"""
import numpy as np
import pytest

from models import f3_model, mixing_model, rich_model, toy_model

pytestmark = pytest.mark.gpu
RTOL = 1e-10
DEFAULT_TRAILING = 1   # library default: tcgen05 int8 Ozaki trailing update (0 = fp64 DMMA)


def both(sb, orc, builder):
    return builder(sb), builder(orc)


def test_cov_single_kernels(sb, orc):
    rng = np.random.default_rng(1)
    x, y = rng.uniform(0, 8, 301), rng.uniform(0, 8, 77)
    for name in ["SEKernel", "Matern12Kernel", "Matern32Kernel", "Matern52Kernel", "WhiteKernel"]:
        fs = sb.gppp(lambda GP: dict(f=GP(getattr(sb, name)())))
        fo = orc.gppp(lambda GP: dict(f=GP(getattr(orc, name)())))
        xs = np.concatenate([x, x[:5]])  # coincident points: k == 1 exactly
        K = sb.cov(fs, sb.GPPPInput("f", xs))
        Ko = orc.cov(fo, orc.GPPPInput("f", xs))
        np.testing.assert_allclose(K, Ko, rtol=0, atol=1e-14)
        assert np.all(np.diag(K) == 1.0)
        assert K[0, 301] == 1.0
        Kxy = sb.cov(fs, sb.GPPPInput("f", x), sb.GPPPInput("f", y))
        np.testing.assert_allclose(Kxy, orc.cov(fo, orc.GPPPInput("f", x), orc.GPPPInput("f", y)), rtol=0, atol=1e-14)
        v = sb.var(fs, sb.GPPPInput("f", x))
        np.testing.assert_array_equal(v, np.ones_like(x))


def test_cov_large_offsets_bitwise_formula(sb, orc):
    """x ~ U(0, 2048): the GEMM-trick distance loses ~1e-9 absolute in d^2; the device must
    follow the same rounding sequence as the CPU path, not the (more accurate) direct form."""
    rng = np.random.default_rng(2)
    x = rng.uniform(0, 2048, 500)
    fs, fo = sb.gppp(lambda GP: dict(f=GP(sb.SEKernel()))), orc.gppp(lambda GP: dict(f=GP(orc.SEKernel())))
    K, Ko = sb.cov(fs, sb.GPPPInput("f", x)), orc.cov(fo, orc.GPPPInput("f", x))
    np.testing.assert_allclose(K, Ko, rtol=4e-16, atol=1e-300)


def test_cov_gppp_blocks(sb, orc):
    rng = np.random.default_rng(3)
    xs = [rng.uniform(-3, 3, n) for n in (130, 61, 259)]
    for builder, names in [(f3_model, ["f1", "f2", "f3"]), (toy_model, ["f3", "f1", "f2"]),
                           (rich_model, ["g1", "g4", "g3"]), (mixing_model, ["g1", "g5", "g3"])]:
        fs, fo = both(sb, orc, builder)
        bs = sb.BlockData(*[sb.GPPPInput(n, x) for n, x in zip(names, xs)])
        bo = orc.BlockData(*[orc.GPPPInput(n, x) for n, x in zip(names, xs)])
        K, Ko = sb.cov(fs, bs), orc.cov(fo, bo)
        np.testing.assert_allclose(K, Ko, rtol=1e-13, atol=1e-14)
        np.testing.assert_allclose(sb.var(fs, bs), orc.var(fo, bo), rtol=1e-13, atol=1e-14)
        np.testing.assert_allclose(sb.mean(fs, bs), orc.mean(fo, bo), rtol=1e-14, atol=1e-15)
        # cross-covariance between different input collections / processes
        b2s, b2o = sb.GPPPInput(names[0], xs[1]), orc.GPPPInput(names[0], xs[1])
        np.testing.assert_allclose(sb.cov(fs, bs, b2s), orc.cov(fo, bo, b2o), rtol=1e-13, atol=1e-14)


def test_cov_multidim(sb, orc):
    rng = np.random.default_rng(4)
    X = rng.standard_normal((3, 150))
    def build(m):
        return m.gppp(lambda GP: (lambda a, b: dict(a=a, b=b, c=m.additive_gp([a, b], [[0, 1], [2]]),
                                                    d=m.stretch(a, np.array([[1., .2, 0], [0, .5, .1]]))))(
            GP(m.SEKernel()), GP(m.Matern32Kernel())))
    fs, fo = build(sb), build(orc)
    for name in ["a", "c", "d"]:
        K = sb.cov(fs, sb.GPPPInput(name, sb.ColVecs(X)))
        Ko = orc.cov(fo, orc.GPPPInput(name, orc.ColVecs(X)))
        np.testing.assert_allclose(K, Ko, rtol=1e-12, atol=1e-13)


@pytest.mark.parametrize("n", [1, 5, 128, 129, 300, 1000])
def test_cholesky_factor(sb, n):
    import scipy.linalg as sla
    rng = np.random.default_rng(n)
    x = np.sort(rng.uniform(0, n / 32 + 1, n))
    fs = sb.gppp(lambda GP: dict(f=GP(sb.SEKernel())))
    fx = fs(sb.GPPPInput("f", x), 0.1)
    L = fx.factor().to_dense_L()
    K = sb.cov(fx)
    Lref = sla.cholesky(K, lower=True)
    np.testing.assert_allclose(L, Lref, rtol=0, atol=1e-12)
    np.testing.assert_allclose(fx.factor().logdet(), 2 * np.sum(np.log(np.diag(Lref))), rtol=1e-12)


@pytest.mark.parametrize("n,ns", [(256, 256), (1000, 333), (4096, 512)])
def test_logpdf_posterior_se(sb, orc, n, ns):
    """Config 1 (N=256) and larger: logpdf + posterior mean/var, rtol 1e-10."""
    rng = np.random.default_rng(123456)
    x = np.sort(rng.uniform(0, n / 32, n))
    xs = rng.uniform(0, n / 32, ns)
    y = np.sin(x) + 0.3 * rng.standard_normal(n)
    fs, fo = sb.gppp(lambda GP: dict(f=GP(sb.SEKernel()))), orc.gppp(lambda GP: dict(f=GP(orc.SEKernel())))
    fxs, fxo = fs(sb.GPPPInput("f", x), 0.1), fo(orc.GPPPInput("f", x), 0.1)
    lp, lpo = sb.logpdf(fxs, y), orc.logpdf(fxo, y)
    np.testing.assert_allclose(lp, lpo, rtol=RTOL)
    Y = np.stack([y, y[::-1], 2 * y], axis=1)
    np.testing.assert_allclose(sb.logpdf(fxs, Y), orc.logpdf(fxo, Y), rtol=RTOL)
    ps, po = sb.posterior(fxs, y), orc.posterior(fxo, y)
    np.testing.assert_allclose(ps.alpha, po.alpha, rtol=1e-8, atol=1e-9)
    m, v = sb.mean_and_var(ps, sb.GPPPInput("f", xs))
    mo, vo = orc.mean_and_var(po, orc.GPPPInput("f", xs))
    np.testing.assert_allclose(m, mo, rtol=RTOL, atol=1e-11)
    np.testing.assert_allclose(v, vo, rtol=RTOL, atol=1e-11)
    mm, sd = sb.marginals(ps(sb.GPPPInput("f", xs), 0.01))
    np.testing.assert_allclose(sd, np.sqrt(vo + 0.01), rtol=RTOL)


def test_logpdf_posterior_gppp(sb, orc):
    """Config-3 shaped: observe f1, f2, f3 = f1 + f2 jointly, predict all three."""
    rng = np.random.default_rng(7)
    ns = (700, 513, 300)
    xs = [rng.uniform(0, 20, n) for n in ns]
    xp = [rng.uniform(0, 20, 90) for _ in range(3)]
    fs, fo = both(sb, orc, f3_model)
    names = ["f1", "f2", "f3"]
    bs, bo = sb.BlockData(*[sb.GPPPInput(n, x) for n, x in zip(names, xs)]), orc.BlockData(*[orc.GPPPInput(n, x) for n, x in zip(names, xs)])
    ps_in, po_in = sb.BlockData(*[sb.GPPPInput(n, x) for n, x in zip(names, xp)]), orc.BlockData(*[orc.GPPPInput(n, x) for n, x in zip(names, xp)])
    fxo = fo(bo, 0.1)
    y = orc.rand(fxo, rng.standard_normal(sum(ns)))
    fxs = fs(bs, 0.1)
    np.testing.assert_allclose(sb.logpdf(fxs, y), orc.logpdf(fxo, y), rtol=RTOL)
    ps, po = sb.posterior(fxs, y), orc.posterior(fxo, y)
    m, v = sb.mean_and_var(ps, ps_in)
    mo, vo = orc.mean_and_var(po, po_in)
    np.testing.assert_allclose(m, mo, rtol=RTOL, atol=1e-10)
    np.testing.assert_allclose(v, vo, rtol=1e-9, atol=1e-10)
    C = sb.cov(ps, ps_in)
    np.testing.assert_allclose(C, orc.cov(po, po_in), rtol=1e-9, atol=1e-10)
    parts = sb.split(ps_in, m)
    assert [len(p) for p in parts] == [90, 90, 90]


def test_rich_model_logpdf_vector_noise(sb, orc):
    rng = np.random.default_rng(8)
    fs, fo = both(sb, orc, rich_model)
    xs = [rng.uniform(-2, 2, n) for n in (200, 150, 141)]
    names = ["g4", "g3", "f2"]
    bs, bo = sb.BlockData(*[sb.GPPPInput(n, x) for n, x in zip(names, xs)]), orc.BlockData(*[orc.GPPPInput(n, x) for n, x in zip(names, xs)])
    noise = rng.uniform(0.05, 0.2, 491)
    fxs, fxo = fs(bs, noise), fo(bo, noise)
    y = orc.rand(fxo, rng.standard_normal(491))
    np.testing.assert_allclose(sb.logpdf(fxs, y), orc.logpdf(fxo, y), rtol=RTOL)
    ys = sb.rand(fxs, np.ones(491))
    np.testing.assert_allclose(ys, orc.rand(fxo, np.ones(491)), rtol=1e-9, atol=1e-9)


def test_not_positive_definite(sb):
    x = np.concatenate([np.linspace(0, 1, 200), np.linspace(0, 1, 200)])  # duplicated points, no noise
    fs = sb.gppp(lambda GP: dict(f=GP(sb.SEKernel())))
    with pytest.raises(sb.PosDefException) as ei:
        sb.logpdf(fs(sb.GPPPInput("f", x), 0.0), np.zeros(400))
    assert 1 <= ei.value.info <= 400


def test_factorisation_is_race_free_and_deterministic(sb):
    """Stress the TMA ring of the DMMA kernel: repeated factorisations of the same matrix must be
    bit-identical (a missing generic->async proxy fence once produced rare stale-operand reads)."""
    rng = np.random.default_rng(99)
    n = 2048
    x = rng.uniform(0, n / 32, n)
    y = rng.standard_normal(n)
    f = sb.gppp(lambda GP: dict(f=GP(sb.SEKernel())))
    ref = None
    for _ in range(25):
        fac = f(sb.GPPPInput("f", x), 0.1).factor()
        L = fac.to_dense_L()
        if ref is None:
            ref = L
        assert np.array_equal(L, ref)


@pytest.mark.parametrize("n,m", [(700, 50), (5000, 300), (20000, 130)])
def test_vfe_elbo_and_approx_posterior(sb, orc, n, m):
    """elbo / dtc / approximate posterior (AbstractGPs VFE via src/gp/sparse_finite_gp.jl:52-62)."""
    rng = np.random.default_rng(n + m)
    x = rng.uniform(0, 30, n)
    z = np.linspace(0, 30, m)
    xs = rng.uniform(0, 30, 150)
    y = np.sin(x) + 0.3 * rng.standard_normal(n)
    noise = rng.uniform(0.05, 0.15, n) if n == 700 else 0.1
    fs, fo = sb.gppp(lambda GP: dict(f=GP(sb.SEKernel()))), orc.gppp(lambda GP: dict(f=GP(orc.SEKernel())))
    fxs, fzs = fs(sb.GPPPInput("f", x), noise), fs(sb.GPPPInput("f", z), 1e-6)
    fxo, fzo = fo(orc.GPPPInput("f", x), noise), fo(orc.GPPPInput("f", z), 1e-6)
    e, eo = sb.elbo(sb.VFE(fzs), fxs, y), orc.elbo(orc.VFE(fzo), fxo, y)
    np.testing.assert_allclose(e, eo, rtol=1e-9)
    np.testing.assert_allclose(sb.dtc(sb.VFE(fzs), fxs, y), orc.dtc(orc.VFE(fzo), fxo, y), rtol=1e-9)
    sp = sb.SparseFiniteGP(fxs, fzs)
    np.testing.assert_allclose(sb.logpdf(sp, y), sb.elbo(sp, y), rtol=1e-13)  # atomics: last-ulp run-to-run
    ps, po = sb.posterior(sp, y), orc.posterior(orc.SparseFiniteGP(fxo, fzo), y)
    mm, vv = sb.mean_and_var(ps, sb.GPPPInput("f", xs))
    np.testing.assert_allclose(mm, orc.mean(po, orc.GPPPInput("f", xs)), rtol=1e-7, atol=1e-8)
    np.testing.assert_allclose(vv, orc.var(po, orc.GPPPInput("f", xs)), rtol=1e-6, atol=1e-8)


@pytest.mark.parametrize("trailing", [0, 1])
@pytest.mark.parametrize("n,m", [(20000, 1024), (40000, 4096)])
def test_vfe_large_m_config4_shape(sb, orc, n, m, trailing):
    """Config-4 geometry (pseudo-points on a unit grid in the observed process, jitter 1e-9 on K_uu,
    x ~ U(0, M), sigma^2 = 0.1) at M = 1024 / 4096: multi-block M x M factors (8 / 32 blocks), several
    16384-row observation chunks; elbo, dtc and the approximate posterior against the oracle, on both
    the DMMA and the tcgen05 paths."""
    rng = np.random.default_rng(n + m)
    x = rng.uniform(0, m, n)
    z = np.arange(m) + 0.5
    xs = rng.uniform(0, m, 200)
    y = np.sin(x) + 0.3 * rng.standard_normal(n)
    fs, fo = sb.gppp(lambda GP: dict(f=GP(sb.SEKernel()))), orc.gppp(lambda GP: dict(f=GP(orc.SEKernel())))
    fxo, fzo = fo(orc.GPPPInput("f", x), 0.1), fo(orc.GPPPInput("f", z), 1e-9)
    eo, do = orc.elbo(orc.VFE(fzo), fxo, y), orc.dtc(orc.VFE(fzo), fxo, y)
    po = orc.vfe_posterior(orc.VFE(fzo), fxo, y)
    ctx = sb.default_context()
    ctx.set_option("trailing", trailing)
    try:
        fxs, fzs = fs(sb.GPPPInput("f", x), 0.1), fs(sb.GPPPInput("f", z), 1e-9)
        ap = sb.approx_posterior(sb.VFE(fzs), fxs, y)
        np.testing.assert_allclose(ap.elbo, eo, rtol=1e-9)
        np.testing.assert_allclose(ap.dtc, do, rtol=1e-9)
        mm, vv = sb.mean_and_var(ap, sb.GPPPInput("f", xs))
        np.testing.assert_allclose(mm, orc.mean(po, orc.GPPPInput("f", xs)), rtol=1e-7, atol=1e-8)
        np.testing.assert_allclose(vv, orc.var(po, orc.GPPPInput("f", xs)), rtol=1e-6, atol=1e-8)
    finally:
        ctx.set_option("trailing", DEFAULT_TRAILING)


def test_vfe_relations(sb):
    """README.md:75-78: pseudo-points == observations => elbo == logpdf; and logpdf > elbo
    (test/gp/sparse_finite_gp.jl:40-41)."""
    rng = np.random.default_rng(77)
    x = rng.uniform(0, 5, 300)
    y = np.sin(x) + 0.3 * rng.standard_normal(300)
    f = sb.gppp(lambda GP: dict(f=GP(sb.Matern32Kernel())))
    fx = f(sb.GPPPInput("f", x), 0.1)
    lp = sb.logpdf(fx, y)
    assert abs(sb.elbo(sb.VFE(f(sb.GPPPInput("f", x), 1e-10)), fx, y) - lp) < 1e-5 * abs(lp)
    assert lp > sb.elbo(sb.VFE(f(sb.GPPPInput("f", x[::10]), 1e-9)), fx, y)


def test_vfe_pseudo_points_in_other_processes(sb, orc):
    """examples/gppp_and_pseudo_points/script.jl:114-121: observe f3 = f1 + f2, pseudo-points in f1 and f2."""
    rng = np.random.default_rng(5)
    fs, fo = both(sb, orc, f3_model)
    x = rng.uniform(0, 10, 900)
    z = np.linspace(0, 10, 40)
    y = rng.standard_normal(900)
    zs = sb.BlockData(sb.GPPPInput("f1", z), sb.GPPPInput("f2", z))
    zo = orc.BlockData(orc.GPPPInput("f1", z), orc.GPPPInput("f2", z))
    e = sb.elbo(sb.VFE(fs(zs, 1e-6)), fs(sb.GPPPInput("f3", x), 0.2), y)
    eo = orc.elbo(orc.VFE(fo(zo, 1e-6)), fo(orc.GPPPInput("f3", x), 0.2), y)
    np.testing.assert_allclose(e, eo, rtol=1e-9)


def _residual_identity(sb, f, obs, y, sub, sigma2):
    """Size-independent check of the whole pipeline at full BASELINE sizes:
    (K + s2 I) alpha = delta  =>  K[sub, :] alpha = delta[sub] - s2 alpha[sub], where the left side
    is the posterior mean evaluated AT a subset of the training inputs (zero-mean prior).
    Also: logpdf's quadratic form |L^{-1} delta|^2 must equal delta' alpha (two different sweeps),
    i.e. logpdf == -(N log 2pi + logdet + y'alpha)/2 with the handle's own logdet."""
    fx = f(obs, sigma2)
    post = sb.posterior(fx, y)
    alpha = post.alpha
    m = sb.mean(post, sub["inputs"])
    rhs = y[sub["idx"]] - sigma2 * alpha[sub["idx"]]
    np.testing.assert_allclose(m, rhs, rtol=0, atol=1e-9 * max(1.0, np.abs(y).max()))
    lp = sb.logpdf(fx, y)
    ld = fx.factor().logdet()
    n = len(y)
    lp2 = -(n * np.log(2 * np.pi) + ld + float(y @ alpha)) / 2
    assert abs(lp - lp2) <= 1e-11 * abs(lp), (lp, lp2)
    # bounds: lambda_min >= s2, and Hadamard: logdet <= sum log diag(K + s2 I)
    assert n * np.log(sigma2) < ld <= float(np.sum(np.log(sb.var(fx)))) + 1e-9 * n
    return lp


@pytest.mark.parametrize("n", [16384, 32768])
def test_config2_oracle_parity_large(sb, n):
    """Config-2 inputs (bench.make_inputs) against the CPU oracle fast path at N = 16384 / 32768:
    logpdf, posterior mean and variance to rtol 1e-10 (north_star tolerance).  The oracle's results
    are stored in tests/golden/config2_oracle.json (written by tests/golden/make_config2_oracle.py):
    at N = 32768 computing them takes minutes and ~35 GB of host memory."""
    import json
    import os
    import bench
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "config2_oracle.json")) as fh:
        gd = json.load(fh)[str(n)]
    assert gd["sigma2"] == bench.SIGMA2
    ns = gd["ns"]
    x, y, xs = bench.make_inputs(n, ns)
    lpo, mo, vo = gd["logpdf"], np.array(gd["mean"]), np.array(gd["var"])
    f = sb.gppp(lambda GP: dict(f=GP(sb.SEKernel())))
    fx = f(sb.GPPPInput("f", x), bench.SIGMA2)
    lp = sb.logpdf(fx, y)
    m, v = sb.mean_and_var(sb.posterior(fx, y), sb.GPPPInput("f", xs))
    assert abs(lp - lpo) <= RTOL * abs(lpo), (lp, lpo)
    np.testing.assert_allclose(m, mo, rtol=RTOL, atol=1e-11)
    np.testing.assert_allclose(v, vo, rtol=RTOL, atol=1e-11)


def test_config3_oracle_parity_3x4096(sb, orc):
    """Config-3 shape (GPPP f3 = f1 + f2 over BlockData) at 3 x 4096 against the oracle's
    recursive routing + LAPACK: logpdf, posterior mean/var of all three processes."""
    rng = np.random.default_rng(123456)
    fs, fo = both(sb, orc, f3_model)
    names = ["f1", "f2", "f3"]
    xs = [rng.uniform(0, 128, 4096) for _ in range(3)]
    xt = [rng.uniform(0, 128, 200) for _ in range(3)]
    bs = sb.BlockData(*[sb.GPPPInput(nm, v) for nm, v in zip(names, xs)])
    bo = orc.BlockData(*[orc.GPPPInput(nm, v) for nm, v in zip(names, xs)])
    ts = sb.BlockData(*[sb.GPPPInput(nm, v) for nm, v in zip(names, xt)])
    to = orc.BlockData(*[orc.GPPPInput(nm, v) for nm, v in zip(names, xt)])
    y = np.concatenate([np.sin(v) for v in xs]) + 0.3 * rng.standard_normal(3 * 4096)
    lp, lpo = sb.logpdf(fs(bs, 0.1), y), orc.logpdf(fo(bo, 0.1), y)
    assert abs(lp - lpo) <= RTOL * abs(lpo), (lp, lpo)
    m, v = sb.mean_and_var(sb.posterior(fs(bs, 0.1), y), ts)
    mo, vo = orc.mean_and_var(orc.posterior(fo(bo, 0.1), y), to)
    np.testing.assert_allclose(m, mo, rtol=RTOL, atol=1e-11)
    np.testing.assert_allclose(v, vo, rtol=RTOL, atol=1e-11)


def test_config2_full_size_properties(sb):
    """BASELINE config 2: SEKernel GP, N=65536 fp64 (bench.py's exact inputs)."""
    import bench
    n = 65536
    x, y, _ = bench.make_inputs(n, 16)
    f = sb.gppp(lambda GP: dict(f=GP(sb.SEKernel())))
    idx = np.arange(0, n, 173)
    lp = _residual_identity(sb, f, sb.GPPPInput("f", x), y, dict(idx=idx, inputs=sb.GPPPInput("f", x[idx])), 0.1)
    assert -1e6 < lp < 0


def test_config2_full_size_tcgen05_vs_dmma(sb):
    """BASELINE config 2 at full size (N = 65536): the two independent implementations of the O(N^3)
    -- fp64 DMMA and tcgen05 int8 Ozaki slices -- must agree on logpdf and on the posterior mean /
    variance at 4096 test points to the north-star tolerance (rtol 1e-10)."""
    import bench
    n, ns = 65536, 4096
    x, y, xs = bench.make_inputs(n, ns)
    f = sb.gppp(lambda GP: dict(f=GP(sb.SEKernel())))
    ctx = sb.default_context()
    res = {}
    try:
        for mode in (0, 1):
            ctx.set_option("trailing", mode)
            ctx.timings(reset=True)
            fx = f(sb.GPPPInput("f", x), bench.SIGMA2)
            lp = sb.logpdf(fx, y)
            m, v = sb.mean_and_var(sb.posterior(fx, y), sb.GPPPInput("f", xs))
            res[mode] = (lp, m, v, ctx.timings()["trailing_int8_ops"])
            del fx
    finally:
        ctx.set_option("trailing", DEFAULT_TRAILING)
    assert res[0][3] == 0 and res[1][3] > 0
    assert abs(res[0][0] - res[1][0]) <= RTOL * abs(res[0][0]), (res[0][0], res[1][0])
    np.testing.assert_allclose(res[1][1], res[0][1], rtol=RTOL, atol=1e-11)
    np.testing.assert_allclose(res[1][2], res[0][2], rtol=RTOL, atol=1e-11)


def test_config3_full_size_properties(sb):
    """BASELINE config 3: GPPP f3 = f1 + f2 over BlockData, 3 x 16384 inputs (N = 49152)."""
    rng = np.random.default_rng(123456)
    xs = [rng.uniform(0, 512, 16384) for _ in range(3)]
    y = rng.standard_normal(49152)
    f = f3_model(sb)
    names = ["f1", "f2", "f3"]
    obs = sb.BlockData(*[sb.GPPPInput(nm, x) for nm, x in zip(names, xs)])
    # subset: every 97th point of every block, addressed through the same BlockData structure
    sel = [np.arange(0, 16384, 97) for _ in range(3)]
    idx = np.concatenate([s + 16384 * b for b, s in enumerate(sel)])
    sub = sb.BlockData(*[sb.GPPPInput(nm, x[s]) for nm, x, s in zip(names, xs, sel)])
    _residual_identity(sb, f, obs, y, dict(idx=idx, inputs=sub), 0.1)
    parts = sb.split(obs, y)
    assert [len(p) for p in parts] == [16384] * 3 and np.array_equal(parts[2], y[32768:])


def test_posterior_finite_gp_rand_and_logpdf(sb, orc):
    """rand / logpdf of a POSTERIOR FiniteGP (README.md:96, examples/process_decomposition/script.jl:36)."""
    rng = np.random.default_rng(21)
    fs, fo = both(sb, orc, f3_model)
    x = rng.uniform(0, 10, 400)
    y = rng.standard_normal(400)
    names = ["f1", "f2", "f3"]
    xs = [rng.uniform(0, 10, n) for n in (50, 37, 64)]
    ps = sb.posterior(fs(sb.GPPPInput("f3", x), 0.1), y)
    po = orc.posterior(fo(orc.GPPPInput("f3", x), 0.1), y)
    bs = sb.BlockData(*[sb.GPPPInput(n, v) for n, v in zip(names, xs)])
    bo = orc.BlockData(*[orc.GPPPInput(n, v) for n, v in zip(names, xs)])
    Z = rng.standard_normal((151, 3))
    for noise in (1e-6, rng.uniform(0.01, 0.02, 151)):
        Ys, Yo = sb.rand(ps(bs, noise), Z), orc.rand(po(bo, noise), Z)
        np.testing.assert_allclose(Ys, Yo, rtol=1e-7, atol=1e-8)
        np.testing.assert_allclose(sb.logpdf(ps(bs, noise), Yo[:, 0]), orc.logpdf(po(bo, noise), Yo[:, 0]), rtol=1e-8)
    f1, f2, f3 = sb.split(bs, Ys)
    assert f1.shape == (50, 3) and f3.shape == (64, 3)


def test_dense_observation_noise(sb, orc):
    """Dense PSD Sigma_y (test/affine_transformations/test_util.jl:114-120)."""
    rng = np.random.default_rng(31)
    n = 333
    x = rng.uniform(0, 10, n)
    A = rng.standard_normal((n, 5))
    S = 0.05 * np.eye(n) + 0.02 * A @ A.T
    y = rng.standard_normal(n)
    fs, fo = both(sb, orc, toy_model)
    fxs, fxo = fs(sb.GPPPInput("f3", x), S), fo(orc.GPPPInput("f3", x), S)
    np.testing.assert_allclose(sb.logpdf(fxs, y), orc.logpdf(fxo, y), rtol=RTOL)
    np.testing.assert_allclose(sb.cov(fxs), orc.cov(fxo), rtol=1e-13, atol=1e-14)
    m, v = sb.mean_and_var(sb.posterior(fxs, y), sb.GPPPInput("f1", x[:40]))
    mo, vo = orc.mean_and_var(orc.posterior(fxo, y), orc.GPPPInput("f1", x[:40]))
    np.testing.assert_allclose(m, mo, rtol=1e-9, atol=1e-10)
    np.testing.assert_allclose(v, vo, rtol=1e-9, atol=1e-10)


def test_nested_gppp_on_device(sb, orc):
    """A GPPP used as an atomic inside another GPPP (gppp.jl test :107-120), through the CUDA path."""
    rng = np.random.default_rng(32)

    def build(m):
        inner = toy_model(m)
        gpc = m.GPC()
        f1 = m.atomic(inner, gpc)
        return m.GPPP(dict(f1=f1, f2=5 * f1), gpc)

    fs, fo = build(sb), build(orc)
    x0, x1 = rng.standard_normal(50), rng.standard_normal(40)
    a_s, b_s = sb.GPPPInput("f1", sb.GPPPInput("f3", x0)), sb.GPPPInput("f2", sb.GPPPInput("f1", x1))
    a_o, b_o = orc.GPPPInput("f1", orc.GPPPInput("f3", x0)), orc.GPPPInput("f2", orc.GPPPInput("f1", x1))
    np.testing.assert_allclose(sb.cov(fs, a_s, b_s), orc.cov(fo, a_o, b_o), rtol=1e-13, atol=1e-14)
    y = rng.standard_normal(50)
    np.testing.assert_allclose(sb.logpdf(fs(a_s, 0.1), y), orc.logpdf(fo(a_o, 0.1), y), rtol=RTOL)


def test_two_posteriors_share_one_factor(sb, orc):
    """posterior is a pure function (AbstractGPs PosteriorGP owns its alpha): a second
    posterior(fx, y2) must not change what the first one predicts (ADVICE r1)."""
    rng = np.random.default_rng(21)
    n = 700
    x, xs = rng.uniform(0, 20, n), rng.uniform(0, 20, 90)
    y1 = np.sin(x) + 0.3 * rng.standard_normal(n)
    y2 = np.cos(2 * x) + 0.3 * rng.standard_normal(n)
    fs, fo = sb.gppp(lambda GP: dict(f=GP(sb.SEKernel()))), orc.gppp(lambda GP: dict(f=GP(orc.SEKernel())))
    fxs, fxo = fs(sb.GPPPInput("f", x), 0.1), fo(orc.GPPPInput("f", x), 0.1)
    p1, p2 = sb.posterior(fxs, y1), sb.posterior(fxs, y2)
    o1, o2 = orc.posterior(fxo, y1), orc.posterior(fxo, y2)
    xi_s, xi_o = sb.GPPPInput("f", xs), orc.GPPPInput("f", xs)
    for p, o in [(p1, o1), (p2, o2), (p1, o1)]:  # interleaved: alpha is re-installed on demand
        np.testing.assert_allclose(sb.mean(p, xi_s), orc.mean(o, xi_o), rtol=RTOL, atol=1e-11)
    np.testing.assert_allclose(p1.alpha, o1.alpha, rtol=1e-9, atol=1e-11)
    np.testing.assert_allclose(p2.alpha, o2.alpha, rtol=1e-9, atol=1e-11)


def test_posterior_cross_cov_and_dense_post_noise(sb, orc):
    """cov(f_post, x, z) with x != z (AbstractGPs App. A) and rand/logpdf of f_post(x*, Sigma_dense)."""
    rng = np.random.default_rng(22)
    fs, fo = both(sb, orc, f3_model)
    xtr = [rng.uniform(0, 10, k) for k in (150, 120, 90)]
    bs = sb.BlockData(*[sb.GPPPInput(nm, v) for nm, v in zip(["f1", "f2", "f3"], xtr)])
    bo = orc.BlockData(*[orc.GPPPInput(nm, v) for nm, v in zip(["f1", "f2", "f3"], xtr)])
    y = orc.rand(fo(bo, 0.1), rng.standard_normal(360))
    ps, po = sb.posterior(fs(bs, 0.1), y), orc.posterior(fo(bo, 0.1), y)
    xa, xb = rng.uniform(0, 10, 41), rng.uniform(0, 10, 57)
    K = sb.cov(ps, sb.GPPPInput("f3", xa), sb.GPPPInput("f1", xb))
    Ko = orc.cov(po, orc.GPPPInput("f3", xa), orc.GPPPInput("f1", xb))
    assert K.shape == (41, 57)
    np.testing.assert_allclose(K, Ko, rtol=1e-9, atol=1e-11)
    # dense observation noise on the posterior FiniteGP
    A = rng.standard_normal((41, 41))
    S = 0.05 * (A @ A.T) / 41 + 0.1 * np.eye(41)
    z = rng.standard_normal(41)
    fps, fpo = ps(sb.GPPPInput("f3", xa), S), po(orc.GPPPInput("f3", xa), S)
    ys = orc.rand(fpo, z)
    np.testing.assert_allclose(sb.rand(fps, z), ys, rtol=1e-8, atol=1e-9)
    lp, lpo = sb.logpdf(fps, ys), orc.logpdf(fpo, ys)
    assert abs(lp - lpo) <= 1e-9 * abs(lpo)


def test_posterior_of_posterior(sb, orc):
    """posterior(f_post(x2, s2), y2) == conditioning the prior on the stacked observations."""
    rng = np.random.default_rng(23)
    fs, fo = sb.gppp(lambda GP: dict(f=GP(sb.Matern52Kernel()))), orc.gppp(lambda GP: dict(f=GP(orc.Matern52Kernel())))
    x1, x2, xs = rng.uniform(0, 10, 200), rng.uniform(0, 10, 130), rng.uniform(0, 10, 50)
    y1, y2 = np.sin(x1), np.sin(x2) + 0.1
    p1 = sb.posterior(fs(sb.GPPPInput("f", x1), 0.1), y1)
    p12 = sb.posterior(p1(sb.GPPPInput("f", x2), 0.2), y2)
    bo = orc.BlockData(orc.GPPPInput("f", x1), orc.GPPPInput("f", x2))
    noise = np.concatenate([np.full(200, 0.1), np.full(130, 0.2)])
    po = orc.posterior(fo(bo, noise), np.concatenate([y1, y2]))
    m, v = sb.mean_and_var(p12, sb.GPPPInput("f", xs))
    mo, vo = orc.mean_and_var(po, orc.GPPPInput("f", xs))
    np.testing.assert_allclose(m, mo, rtol=RTOL, atol=1e-11)
    np.testing.assert_allclose(v, vo, rtol=1e-9, atol=1e-11)


def test_vfe_approx_posterior_cov(sb, orc):
    rng = np.random.default_rng(24)
    n, m = 1500, 260
    x = np.sort(rng.uniform(0, 30, n))
    z = np.linspace(0, 30, m)
    y = np.sin(x) + 0.2 * rng.standard_normal(n)
    xs, xz = rng.uniform(0, 30, 70), rng.uniform(0, 30, 33)
    fs, fo = sb.gppp(lambda GP: dict(f=GP(sb.SEKernel()))), orc.gppp(lambda GP: dict(f=GP(orc.SEKernel())))
    aps = sb.approx_posterior(sb.VFE(fs(sb.GPPPInput("f", z), 1e-9)), fs(sb.GPPPInput("f", x), 0.1), y)
    apo = orc.vfe_posterior(orc.VFE(fo(orc.GPPPInput("f", z), 1e-9)), fo(orc.GPPPInput("f", x), 0.1), y)
    K, Ko = sb.cov(aps, sb.GPPPInput("f", xs)), orc.cov(apo, orc.GPPPInput("f", xs))
    np.testing.assert_allclose(K, Ko, rtol=1e-7, atol=1e-9)
    np.testing.assert_allclose(np.diag(K), sb.var(aps, sb.GPPPInput("f", xs)), rtol=1e-7, atol=1e-9)
    Kx = sb.cov(aps, sb.GPPPInput("f", xs), sb.GPPPInput("f", xz))
    np.testing.assert_allclose(Kx, orc.cov(apo, orc.GPPPInput("f", xs), orc.GPPPInput("f", xz)), rtol=1e-7, atol=1e-9)


@pytest.fixture
def ozaki_ctx(sb):
    """Route the trailing updates of the default context through the tcgen05 int8-Ozaki kernel."""
    ctx = sb.default_context()
    ctx.set_option("trailing", 1)
    try:
        yield ctx
    finally:
        ctx.set_option("trailing", DEFAULT_TRAILING)


# Test points per size; the sizes below 2500 end the factorisation with a short outer step:
# nblk = ceil(N / 128) = 9, 10, 11, 13 leaves nq = 1, 2, 3, 1 block columns (1663: N % 128 = 127).
OZ_TEST_POINTS = {1025: 1, 1153: 127, 1281: 129}
OZ_MODES = [0, 2, 4, 6, 8, 10, 16]   # the tcgen05 variants SB_OZ_MODE accepts; 2, 6, 10 factor by look-ahead
OZ_DEFAULT_MODE = 8


@pytest.mark.parametrize("n", [2500, 4096, 1025, 1153, 1281, 1663])
def test_tcgen05_ozaki_trailing_update_parity(sb, orc, ozaki_ctx, n):
    """fp64 Cholesky whose trailing SYRK runs as 28 int8 tcgen05 MMAs per fp64 MMA (ozaki.cu):
    the factor must agree with LAPACK to 1e-12 and logpdf / posterior with the oracle to 1e-10.
    At N = 1153 logpdf and posterior are also checked under every kernel variant (oz_mode)."""
    import scipy.linalg as sla
    rng = np.random.default_rng(41)
    x, xs = rng.uniform(0, n / 32, n), rng.uniform(0, n / 32, OZ_TEST_POINTS.get(n, 300))
    y = np.sin(x) + 0.3 * rng.standard_normal(n)
    fs, fo = sb.gppp(lambda GP: dict(f=GP(sb.SEKernel()))), orc.gppp(lambda GP: dict(f=GP(orc.SEKernel())))
    fxs, fxo = fs(sb.GPPPInput("f", x), 0.1), fo(orc.GPPPInput("f", x), 0.1)
    t0 = ozaki_ctx.timings(reset=True)
    lp, lpo = sb.logpdf(fxs, y), orc.logpdf(fxo, y)
    tm = ozaki_ctx.timings()
    assert tm["trailing_int8_ops"] > 0, "the tcgen05 path did not run"
    assert abs(lp - lpo) <= RTOL * abs(lpo), (lp, lpo)
    L = fxs.factor().to_dense_L()
    Lref = sla.cholesky(orc.cov(fxo), lower=True)
    np.testing.assert_allclose(L, Lref, rtol=0, atol=1e-12)
    m, v = sb.mean_and_var(sb.posterior(fxs, y), sb.GPPPInput("f", xs))
    mo, vo = orc.mean_and_var(orc.posterior(fxo, y), orc.GPPPInput("f", xs))
    np.testing.assert_allclose(m, mo, rtol=RTOL, atol=1e-11)
    np.testing.assert_allclose(v, vo, rtol=RTOL, atol=1e-11)
    if n != 1153:
        return
    try:
        for mode in OZ_MODES:
            ozaki_ctx.set_option("oz_mode", mode)
            ozaki_ctx.timings(reset=True)
            fxm = fs(sb.GPPPInput("f", x), 0.1)
            lp = sb.logpdf(fxm, y)
            assert ozaki_ctx.timings()["trailing_int8_ops"] > 0, f"oz_mode {mode}: the tcgen05 path did not run"
            assert abs(lp - lpo) <= RTOL * abs(lpo), (mode, lp, lpo)
            m, v = sb.mean_and_var(sb.posterior(fxm, y), sb.GPPPInput("f", xs))
            np.testing.assert_allclose(m, mo, rtol=RTOL, atol=1e-11, err_msg=f"oz_mode {mode}")
            np.testing.assert_allclose(v, vo, rtol=RTOL, atol=1e-11, err_msg=f"oz_mode {mode}")
    finally:
        ozaki_ctx.set_option("oz_mode", OZ_DEFAULT_MODE)


def test_dmma_trailing_update_parity(sb, orc):
    """The fp64 DMMA path (SB_TRAILING=dmma / option trailing=0) stays covered now that tcgen05 is the default."""
    import scipy.linalg as sla
    rng = np.random.default_rng(43)
    n = 3000
    x, xs = rng.uniform(0, n / 32, n), rng.uniform(0, n / 32, 100)
    y = np.sin(x) + 0.3 * rng.standard_normal(n)
    fs, fo = sb.gppp(lambda GP: dict(f=GP(sb.SEKernel()))), orc.gppp(lambda GP: dict(f=GP(orc.SEKernel())))
    ctx = sb.default_context()
    ctx.set_option("trailing", 0)
    try:
        fxs, fxo = fs(sb.GPPPInput("f", x), 0.1), fo(orc.GPPPInput("f", x), 0.1)
        ctx.timings(reset=True)
        lp, lpo = sb.logpdf(fxs, y), orc.logpdf(fxo, y)
        assert ctx.timings()["trailing_int8_ops"] == 0
        assert abs(lp - lpo) <= RTOL * abs(lpo)
        np.testing.assert_allclose(fxs.factor().to_dense_L(), sla.cholesky(orc.cov(fxo), lower=True), rtol=0, atol=1e-12)
        m, v = sb.mean_and_var(sb.posterior(fxs, y), sb.GPPPInput("f", xs))
        mo, vo = orc.mean_and_var(orc.posterior(fxo, y), orc.GPPPInput("f", xs))
        np.testing.assert_allclose(m, mo, rtol=RTOL, atol=1e-11)
        np.testing.assert_allclose(v, vo, rtol=RTOL, atol=1e-11)
    finally:
        ctx.set_option("trailing", DEFAULT_TRAILING)


def test_tcgen05_ozaki_gppp_badly_scaled_rows(sb, orc, ozaki_ctx):
    """Rows of very different magnitude (function-scaled processes, heteroscedastic noise): the per-row
    power-of-two scaling of the digit planes must keep fp64-level accuracy."""
    rng = np.random.default_rng(42)
    fs, fo = both(sb, orc, rich_model)
    names = ["g1", "g4", "g3"]
    xs = [rng.uniform(-3, 3, k) for k in (900, 700, 800)]
    bs = sb.BlockData(*[sb.GPPPInput(nm, v) for nm, v in zip(names, xs)])
    bo = orc.BlockData(*[orc.GPPPInput(nm, v) for nm, v in zip(names, xs)])
    noise = 10.0 ** rng.uniform(-4, 0, 2400)
    y = orc.rand(fo(bo, noise), rng.standard_normal(2400))
    lp, lpo = sb.logpdf(fs(bs, noise), y), orc.logpdf(fo(bo, noise), y)
    assert ozaki_ctx.timings()["trailing_int8_ops"] > 0
    assert abs(lp - lpo) <= 1e-9 * abs(lpo), (lp, lpo)


def test_factor_export_import_roundtrip(sb, orc):
    """Checkpoint / resume of the device-resident factor (SURVEY 8f.4): an imported handle must
    reproduce logpdf and the posterior bit for bit."""
    rng = np.random.default_rng(51)
    n = 1500
    x, xs = rng.uniform(0, 40, n), rng.uniform(0, 40, 64)
    y = np.sin(x) + 0.3 * rng.standard_normal(n)
    f = sb.gppp(lambda GP: dict(f=GP(sb.Matern32Kernel())))
    fx = f(sb.GPPPInput("f", x), 0.1)
    lp = sb.logpdf(fx, y)
    post = sb.posterior(fx, y)
    m, v = sb.mean_and_var(post, sb.GPPPInput("f", xs))
    blob = sb.save_factor(fx)
    assert blob.dtype == np.uint8 and blob.size > n * (n + 128) // 2 * 8
    fx2 = sb.load_factor(f(sb.GPPPInput("f", x), 0.1), blob.copy())
    assert sb.logpdf(fx2, y) == lp
    m2, v2 = sb.mean_and_var(sb.posterior(fx2, y), sb.GPPPInput("f", xs))
    np.testing.assert_array_equal(m2, m)
    np.testing.assert_array_equal(v2, v)
    with pytest.raises(sb.SthenoB200Error):
        sb.load_factor(f(sb.GPPPInput("f", x), 0.1), blob[:1000].copy())


def test_logpdf_gradients_vs_finite_differences(sb, orc):
    """SURVEY 8f.1: d logpdf / d (kernel variances, lengthscales, noise) from the device
    (1/2 tr((aa' - K^-1) dK)) against central finite differences of the ORACLE's logpdf
    (the reference checks AD against FiniteDifferences at 1e-4, test/affine_transformations/test_util.jl:31)."""
    rng = np.random.default_rng(61)
    x3, x1 = rng.uniform(0, 10, 300), rng.uniform(0, 10, 220)
    y = rng.standard_normal(520)

    def build(m, th):
        v1, l1, v2, l2 = th[:4]
        def mk(GP):
            f1 = GP(v1 * m.with_lengthscale(m.SEKernel(), l1))
            f2 = GP(v2 * m.with_lengthscale(m.Matern52Kernel(), l2) + 0.05 * m.WhiteKernel())
            return dict(f1=f1, f2=f2, f3=f1 + 0.5 * f2)
        return m.gppp(mk)

    def obs(m):
        return m.BlockData(m.GPPPInput("f3", x3), m.GPPPInput("f1", x1))

    th = np.array([1.3, 0.8, 0.6, 1.7, 0.15])
    fs = build(sb, th)
    gr = sb.grad_logpdf(fs(obs(sb), th[4]), y)
    f1, f2 = fs.fs["f1"], fs.fs["f2"]
    k1, k2 = gr.for_atom(f1, 0), gr.for_atom(f2, 0)
    got = np.array([k1["dcoeff"], -k1["dlogscale"] / th[1], k2["dcoeff"], -k2["dlogscale"] / th[3], gr.noise])

    def lp(t):
        return orc.logpdf(build(orc, t)(obs(orc), t[4]), y)

    fd = np.zeros(5)
    for i in range(5):
        h = 1e-5 * th[i]
        tp, tmn = th.copy(), th.copy()
        tp[i] += h
        tmn[i] -= h
        fd[i] = (lp(tp) - lp(tmn)) / (2 * h)
    np.testing.assert_allclose(got, fd, rtol=1e-5, atol=1e-6)
    # White component of f2: d/d(its multiplier); vector noise: per-observation derivative
    kw = gr.for_atom(f2, 1)
    hw = 1e-6

    def lpw(wv):
        def mk(GP):
            f1 = GP(th[0] * orc.with_lengthscale(orc.SEKernel(), th[1]))
            f2 = GP(th[2] * orc.with_lengthscale(orc.Matern52Kernel(), th[3]) + wv * orc.WhiteKernel())
            return dict(f1=f1, f2=f2, f3=f1 + 0.5 * f2)
        return orc.logpdf(orc.gppp(mk)(obs(orc), th[4]), y)

    np.testing.assert_allclose(kw["dcoeff"], (lpw(0.05 + hw) - lpw(0.05 - hw)) / (2 * hw), rtol=1e-5)
    nv = rng.uniform(0.1, 0.3, 520)
    gv = sb.grad_logpdf(fs(obs(sb), nv), y)
    i0 = 17
    nvp, nvm = nv.copy(), nv.copy()
    nvp[i0] += 1e-6
    nvm[i0] -= 1e-6
    fo = build(orc, th)
    fdv = (orc.logpdf(fo(obs(orc), nvp), y) - orc.logpdf(fo(obs(orc), nvm), y)) / 2e-6
    np.testing.assert_allclose(gv.noise[i0], fdv, rtol=1e-5)
