"""GPU parity against the REFERENCE ITSELF: the CUDA engine (through the C ABI) vs src/DESeq2.cpp compiled unchanged into
oracle/_ref/libdeseq2_ref.so (stand-in Rcpp / Armadillo / Rmath headers), whose outputs for these inputs are stored
under tests/golden/reference/ (tests/reference_outputs.py).  Tolerance 1e-6 (north_star); `iter` / `iter_accept` exact
on every gene whose line-search decisions are not knife-edge (the oracle's margin, which
tests/test_oracle_vs_reference.py ties to the same reference build)."""
import numpy as np
import pytest

from helpers import DISP_KEYS, beta_args, disp_args, make_case, rel_err
from reference_outputs import Reference, take

pytestmark = pytest.mark.gpu
TOL = 1e-6


@pytest.fixture
def ref(request):
    return Reference("parity_reference_gpu", request.node.name)


@pytest.mark.parametrize("n,m,seed", [(2500, 100, 211), (2000, 6, 212), (1200, 24, 213)])
def test_fit_disp_vs_reference(engine, oracle, ref, n, m, seed):
    c = make_case(n, m, seed=seed)
    a = disp_args(c, c["mu"], np.log(c["alpha0"]))
    r = ref.fitDisp(**a, nthreads=8)
    g = take(engine.fitDisp(**a), r)
    margin = oracle.fitDisp(**a, with_margin=True)["margin"][r["rows"]]
    robust = margin > 64
    same = (g["iter"] == r["iter"]) & (g["iter_accept"] == r["iter_accept"])
    assert not np.any(~same & robust), np.flatnonzero(~same & robust)[:8]
    sel = same & robust
    assert np.max(rel_err(np.exp(g["log_alpha"][sel]), np.exp(r["log_alpha"][sel]))) < TOL
    for k in ("log_alpha", "initial_lp", "last_lp"):
        assert np.nanmax(rel_err(g[k][sel], r[k][sel])) < TOL, k
    rest = ~sel
    if rest.any():     # knife-edge genes: both end at the same posterior value
        d = np.abs(g["last_lp"][rest] - r["last_lp"][rest]) / (1.0 + np.abs(r["last_lp"][rest]))
        assert np.nanmax(d) < 1e-5


@pytest.mark.parametrize("n,m,seed,useQR", [(2500, 100, 221, True), (2000, 6, 222, True), (1200, 24, 223, False)])
def test_fit_beta_vs_reference(engine, ref, n, m, seed, useQR):
    c = make_case(n, m, seed=seed)
    alpha = np.clip(0.1 + 4.0 / c["baseMean"], 1e-8, 10)
    a = beta_args(c, alpha, useQR=useQR)
    r = ref.fitBeta(**a, nthreads=8)
    g = take(engine.fitBeta(**a), r)
    assert np.array_equal(g["iter"], r["iter"])
    for k in ("beta_mat", "beta_var_mat", "hat_diagonals", "contrast_num", "contrast_denom", "deviance"):
        assert np.nanmax(rel_err(g[k], r[k], floor=1e-8)) < TOL, k
    assert np.nanmax(rel_err(np.sqrt(g["beta_var_mat"]), np.sqrt(r["beta_var_mat"]))) < TOL


def test_fit_beta_weights_ridge_general_p_vs_reference(engine, ref):
    from deseq2_b200 import synth
    m = 40
    x = synth.design_factor(m, 10)
    c = make_case(500, m, x=x, seed=231)
    rng = np.random.default_rng(231)
    w = rng.uniform(0.3, 1.0, c["counts"].shape)
    lam = np.full(10, 1e-6) / np.log(2) ** 2
    lam[-1] = 0.3
    alpha = np.clip(0.1 + 4 / c["baseMean"], 1e-8, m)
    a = beta_args(c, alpha, weights=w, useWeights=True, lam=lam, x=x, contrast=np.r_[np.zeros(9), 1.0])
    r = ref.fitBeta(**a, nthreads=8)
    g = take(engine.fitBeta(**a), r)
    assert np.array_equal(g["iter"], r["iter"])
    for k in ("beta_mat", "beta_var_mat", "hat_diagonals", "contrast_num", "contrast_denom", "deviance"):
        assert np.nanmax(rel_err(g[k], r[k], floor=1e-8)) < TOL, k


def test_fit_disp_grid_vs_reference(engine, ref):
    c = make_case(400, 30, seed=241)
    grid = np.linspace(np.log(1e-8), np.log(30), 20)
    kw = dict(ySEXP=c["counts"], xSEXP=c["x"], mu_hatSEXP=c["mu"], disp_gridSEXP=grid,
              log_alpha_prior_meanSEXP=np.log(0.1 + 4 / c["baseMean"]), log_alpha_prior_sigmasqSEXP=0.5,
              usePriorSEXP=True, weightsSEXP=None, useWeightsSEXP=False, weightThresholdSEXP=1e-2, useCRSEXP=True)
    r = ref.fitDispGrid(**kw, nthreads=4)
    g, r = engine.fitDispGrid(**kw)["log_alpha"][r["rows"]], r["log_alpha"]
    assert np.mean(np.abs(g - r) < 1e-9) > 0.995
    assert np.max(np.abs(g - r)) < 2.0 * (grid[1] - grid[0]) / 9.5
