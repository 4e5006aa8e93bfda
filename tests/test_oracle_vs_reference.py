"""The reference pin (VERDICT r01 #2): the CPU oracle (oracle/nbglm_oracle.c, a restatement) against the REFERENCE'S OWN
translation unit, src/DESeq2.cpp, compiled unchanged into oracle/_ref/libdeseq2_ref.so against stand-in Rcpp /
Armadillo / Rmath headers (oracle/ref_standin/, oracle/Makefile `ref`), whose outputs for these inputs are stored under
tests/golden/reference/ (tests/reference_outputs.py).  All three entry points, weights (incl. Cox-Reid row / column
removal), both useQR branches, ridge, normalisation-factor matrices, maxit = 0, INTSXP and REALSXP counts, the
divergence sentinel of test_optim.R.

Tolerances: fitBeta / fitDispGrid / the posterior and its derivatives are the same formulas evaluated by two
implementations of the same fp64 arithmetic (only the p x p linear algebra and the nmath restatement differ), so they
must agree to 1e-9; fitDisp's control flow (iter, iter_accept) must be IDENTICAL for every gene whose decisions are not
knife-edge (oracle margin > 64 rounding bounds, see oracle_fit_disp)."""
import numpy as np
import pytest

from helpers import DISP_KEYS, beta_args, disp_args, make_case, rel_err
from reference_outputs import Reference, take


@pytest.fixture
def ref(request):
    return Reference("oracle_vs_reference", request.node.name)


TIGHT = 1e-9


def _cmp_disp(o, r, m, name, min_same=0.95):
    o = dict(o, n_samples=m)
    same = (o["iter"] == r["iter"]) & (o["iter_accept"] == r["iter_accept"])
    robust = o["margin"] > 64
    assert not np.any(~same & robust), f"{name}: robust genes differ in control flow: {np.flatnonzero(~same & robust)[:8]}"
    assert same.mean() >= min_same, (name, same.mean())
    # initial values: no control flow involved, every gene
    assert np.nanmax(rel_err(r["initial_lp"], o["initial_lp"])) < TIGHT
    scale = np.abs(o["initial_lp"]) * 1e-3 + 1e-12
    assert np.nanmax(np.abs(r["initial_dlp"] - o["initial_dlp"]) / (scale + np.abs(o["initial_dlp"]))) < 1e-7
    # rounding-noise floor shared by BOTH implementations: every sample contributes lgamma(y + 1/alpha) - lgamma(1/alpha),
    # a difference of numbers of size lgamma(1/alpha) (1.7e9 at alpha = 1e-8, where most m = 6 genes end): 2^-52 of that
    # per sample is the best any fp64 evaluation of the reference's formula can do
    from scipy.special import gammaln
    m = o["n_samples"]
    noise = 16 * 2.0 ** -52 * m * np.abs(gammaln(np.exp(-np.minimum(o["log_alpha"], r["log_alpha"]))))[same]
    for k in DISP_KEYS:
        d = np.maximum(np.abs(r[k][same] - o[k][same]) - (0.0 if k == "log_alpha" else noise), 0.0)
        if k in ("last_dlp", "last_change", "last_d2lp", "initial_dlp"):
            # differences of nearly equal numbers (at alpha -> 1e-8 the trigamma / lgamma terms cancel to rounding
            # noise in BOTH implementations): absolute error on the scale of the posterior
            err = d / (np.abs(o["last_lp"][same]) * 1e-3 + np.abs(o[k][same]) + 1e-12)
            assert np.nanmax(err) < 1e-6, (name, k, np.nanmax(err))
        else:
            assert np.nanmax(d / np.maximum(np.abs(o[k][same]), 1e-12)) < 1e-8, (name, k)
    rest = ~same
    if rest.any():   # knife-edge genes: either branch is a correct fp64 evaluation; same posterior value reached
        d = np.abs(r["last_lp"][rest] - o["last_lp"][rest]) / (1 + np.abs(o["last_lp"][rest]))
        assert np.nanmax(d) < 1e-5, (name, np.nanmax(d))
    return same.mean()


def _disp(oracle, ref, a):
    r = ref.fitDisp(**a)
    return take(oracle.fitDisp(**a, with_margin=True), r), r


def _beta(oracle, ref, a):
    r = ref.fitBeta(**a)
    return take(oracle.fitBeta(**a), r), r


def _cmp_beta(o, r, name):
    assert np.array_equal(o["iter"], r["iter"]), name
    for k in ("beta_mat", "beta_var_mat", "hat_diagonals", "contrast_num", "contrast_denom", "deviance"):
        err = rel_err(r[k], o[k], floor=1e-8)
        assert np.all(np.isnan(r[k]) == np.isnan(o[k])), (name, k)
        assert np.nanmax(err) < TIGHT, (name, k, np.nanmax(err))


@pytest.mark.parametrize("n,m,seed", [(600, 6, 1), (400, 12, 2), (300, 100, 3), (200, 37, 4)])
def test_fit_disp_mle(oracle, ref, n, m, seed):
    c = make_case(n, m, seed=seed)
    a = disp_args(c, c["mu"], np.log(c["alpha0"]))
    _cmp_disp(*_disp(oracle, ref, a), m=a["ySEXP"].shape[1], name=f"mle {n}x{m}", min_same=0.9)


def test_fit_disp_map_prior_and_real_counts(oracle, ref):
    c = make_case(400, 24, seed=5)
    mle = oracle.fitDisp(**disp_args(c, c["mu"], np.log(c["alpha0"])))
    fit = 0.1 + 4.0 / c["baseMean"]
    a = disp_args(c, c["mu"], mle["log_alpha"], prior_mean=np.log(fit), sigmasq=0.6, usePrior=True,
                  y=c["counts"].astype(np.float64))           # REALSXP counts (the INTSXP coercion is the default path)
    _cmp_disp(*_disp(oracle, ref, a), m=a["ySEXP"].shape[1], name="map")
    a = disp_args(c, c["mu"], np.log(c["alpha0"]), useCR=False)
    _cmp_disp(*_disp(oracle, ref, a), m=a["ySEXP"].shape[1], name="noCR", min_same=0.9)


def _weights_for(shape, seed, p_small=0.08):
    rng = np.random.default_rng(seed)
    w = rng.uniform(0.3, 1.0, shape)
    w[rng.random(shape) < p_small] = 1e-3                     # below weightThreshold: row leaves the Cox-Reid term
    return np.maximum(w / w.max(axis=1, keepdims=True), 1e-6)


@pytest.mark.parametrize("design,seed", [("condition", 51), ("batch", 52), ("factor4", 53)])
def test_fit_disp_weights_and_designs(oracle, ref, design, seed):
    from deseq2_b200 import synth
    m = 24
    x = {"condition": synth.design_condition(m), "batch": synth.design_batch_condition(m, 2),
         "factor4": synth.design_factor(m, 4)}[design]
    c = make_case(300, m, x=x, seed=seed)
    alpha = np.clip(0.1 + 4 / c["baseMean"], 1e-8, m)
    mu = c["mu"] if c["mu"] is not None else np.maximum(
        c["nf"] * np.exp(oracle.fitBeta(**beta_args(c, alpha))["beta_mat"] @ x.T), 0.5)
    w = _weights_for(c["counts"].shape, seed)
    a = disp_args(c, mu, np.log(c["alpha0"]), prior_mean=np.log(alpha), sigmasq=0.8, usePrior=True, weights=w,
                  useWeights=True)
    _cmp_disp(*_disp(oracle, ref, a), m=a["ySEXP"].shape[1], name=f"weights/{design}", min_same=0.9)


def test_fit_disp_weights_drop_a_design_column(oracle, ref):
    """src/DESeq2.cpp:41-43: all samples of one group below the threshold -> the column is removed from the CR term."""
    from deseq2_b200 import synth
    m = 12
    c = make_case(150, m, x=synth.design_condition(m), seed=54)
    w = np.ones(c["counts"].shape)
    w[:, m // 2:] = 5e-3
    a = disp_args(c, c["mu"], np.log(c["alpha0"]), weights=w, useWeights=True)
    _cmp_disp(*_disp(oracle, ref, a), m=a["ySEXP"].shape[1], name="dropped column", min_same=0.85)


@pytest.mark.parametrize("usePrior,useWeights", [(True, False), (False, False), (True, True)])
def test_fit_disp_grid(oracle, ref, usePrior, useWeights):
    c = make_case(250, 30, seed=23)
    grid = np.linspace(np.log(1e-8), np.log(30), 20)
    w = _weights_for(c["counts"].shape, 7) if useWeights else None
    kw = dict(ySEXP=c["counts"], xSEXP=c["x"], mu_hatSEXP=c["mu"], disp_gridSEXP=grid,
              log_alpha_prior_meanSEXP=np.log(0.1 + 4 / c["baseMean"]), log_alpha_prior_sigmasqSEXP=0.5,
              usePriorSEXP=usePrior, weightsSEXP=w, useWeightsSEXP=useWeights, weightThresholdSEXP=1e-2, useCRSEXP=True)
    r = ref.fitDispGrid(**kw)
    o, r = oracle.fitDispGrid(**kw)["log_alpha"][r["rows"]], r["log_alpha"]
    assert np.mean(o == r) > 0.99                              # same grid point unless two values tie to rounding
    assert np.max(np.abs(o - r)) < 2.0 * (grid[1] - grid[0]) / 9.5


@pytest.mark.parametrize("n,m,seed,useQR", [(500, 100, 31, True), (500, 6, 32, True), (300, 37, 33, False),
                                            (300, 8, 34, False)])
def test_fit_beta(oracle, ref, n, m, seed, useQR):
    c = make_case(n, m, seed=seed)
    alpha = np.clip(0.1 + 4.0 / c["baseMean"], 1e-8, 10)
    a = beta_args(c, alpha, useQR=useQR)
    _cmp_beta(*_beta(oracle, ref, a), f"beta {n}x{m} qr={useQR}")


@pytest.mark.parametrize("design,seed,useQR", [("batch", 61, True), ("factor4", 62, False), ("intercept", 63, True),
                                               ("factor10", 64, True)])
def test_fit_beta_designs_weights_nf_matrix_ridge(oracle, ref, design, seed, useQR):
    from deseq2_b200 import synth
    m = 40 if design == "factor10" else 24
    x = {"batch": synth.design_batch_condition(m, 2), "factor4": synth.design_factor(m, 4),
         "intercept": np.ones((m, 1)), "factor10": synth.design_factor(m, 10)}[design]
    c = make_case(300, m, x=x if design != "intercept" else None, seed=seed)
    if design == "intercept":
        c["x"] = x
        c["beta0"] = np.log(c["baseMean"])[:, None]
    rng = np.random.default_rng(seed)
    nf = c["nf"] * np.exp(rng.normal(0, 0.2, c["nf"].shape))
    nf /= np.exp(np.mean(np.log(nf), axis=1, keepdims=True))
    alpha = np.clip(0.1 + 4 / c["baseMean"], 1e-8, m)
    w = _weights_for(c["counts"].shape, seed, p_small=0.0)
    p = x.shape[1]
    lam = np.full(p, 1e-6) / np.log(2) ** 2
    if p > 1:
        lam[-1] = 0.3
    a = beta_args(c, alpha, nf=nf, weights=w, useWeights=True, useQR=useQR, lam=lam, x=x,
                  contrast=np.r_[np.zeros(p - 1), 1.0])
    _cmp_beta(*_beta(oracle, ref, a), f"beta/{design}")


def test_fit_beta_maxit0_and_divergence_sentinel(oracle, ref):
    c = make_case(200, 24, seed=34)
    alpha = np.clip(0.1 + 4.0 / c["baseMean"], 1e-8, 10)
    fit = oracle.fitBeta(**beta_args(c, alpha))
    a = beta_args(c, alpha, beta0=fit["beta_mat"], maxit=0, useQR=False, contrast=np.array([0.0, 1.0]))
    o, r = _beta(oracle, ref, a)
    assert np.all(r["iter"] == 0)
    _cmp_beta(o, r, "maxit0")
    # test_optim.R:29-39: the 0/1000 row must report iter == maxit in the reference and in the oracle
    y = np.array([[0, 0, 0, 0, 0, 1000, 1000, 0, 0, 0], [5, 7, 6, 4, 5, 9, 11, 8, 10, 12]], dtype=np.int32)
    x = np.c_[np.ones(10), np.r_[np.zeros(5), np.ones(5)]]
    args = (y, x, np.ones((2, 10)), [0.1, 0.1], [1, 0], np.ones((2, 2)), np.full(2, 1e-6) / np.log(2) ** 2, None,
            False, 1e-8, 100, True, 0.5)
    o, r = oracle.fitBeta(*args), ref.fitBeta(*args)
    assert r["iter"][0] == 100 and r["iter"][1] < 100 and np.array_equal(o["iter"], r["iter"])


def test_standin_nmath_against_mpmath(oracle):
    """The nmath stand-in behind the reference build (oracle/ref_standin/rmath_standin.c) at 40 digits."""
    import ctypes as C
    import os
    import subprocess

    import mpmath as mp
    subprocess.check_call(["make", "-C", os.path.dirname(oracle.__file__), "-s", "librmath_standin.so"])
    L = C.CDLL(os.path.join(os.path.dirname(oracle.__file__), "librmath_standin.so"))
    for f in ("Rf_lgammafn", "Rf_digamma", "Rf_trigamma"):
        getattr(L, f).restype = C.c_double
        getattr(L, f).argtypes = [C.c_double]
    L.Rf_dnbinom_mu.restype = C.c_double
    L.Rf_dnbinom_mu.argtypes = [C.c_double, C.c_double, C.c_double, C.c_int]
    L.R_pow_di.restype = C.c_double
    L.R_pow_di.argtypes = [C.c_double, C.c_int]
    mp.mp.dps = 40
    rng = np.random.default_rng(5)
    for x in np.concatenate([rng.uniform(1e-3, 40, 150), 10 ** rng.uniform(-6, 9, 150)]):
        xm = mp.mpf(float(x))
        for f, g in ((L.Rf_lgammafn, mp.loggamma), (L.Rf_digamma, mp.digamma), (L.Rf_trigamma, lambda t: mp.polygamma(1, t))):
            want = float(g(xm))
            assert abs(f(float(x)) - want) <= 4e-15 * max(1.0, abs(want)), (f, x)
    for _ in range(300):
        size = 10 ** rng.uniform(-2, 9)
        mu = 10 ** rng.uniform(-1, 5)
        k = int(rng.choice([0, 1, 2, 5, rng.poisson(mu)]))
        sm, mm = mp.mpf(size), mp.mpf(mu)
        want = float(mp.loggamma(k + sm) - mp.loggamma(sm) - mp.loggamma(k + 1) + sm * mp.log(sm / (sm + mm))
                     + k * mp.log(mm / (sm + mm)))
        got = L.Rf_dnbinom_mu(float(k), size, mu, 1)
        # R's dbinom_raw route forms size/(size+mu) in double, so its error grows like size * 2^-52 (1e-9 at
        # size = 7e8 -- R's own behaviour, the "FIXME" in nmath/dnbinom.c): compare with the exact value where the
        # published algorithm is accurate, and with the oracle's separate restatement of it everywhere
        if size <= 1e6:
            assert abs(got - want) <= 1e-10 * max(1.0, abs(want)), (k, size, mu, got, want)
        assert abs(got - oracle.dnbinom_mu_log(k, size, mu)) <= 1e-13 * max(1.0, abs(want)), (k, size, mu)
    assert L.R_pow_di(3.0, -2) == 1.0 / 9.0 and L.R_pow_di(2.0, 10) == 1024.0 and L.R_pow_di(5.0, 0) == 1.0
