"""The product's CUDA kernels, executed on the CPU by the SIMT emulator (tests/simt_emu/), against the oracle.

tests/simt_emu/build_emu.py compiles deseq2_b200/csrc/*.cu -- the very sources nvcc compiles for sm_100a, with three
mechanical rewrites (launch syntax, `extern __shared__`, one PTX statement) -- into libb200nb_emu.so, which exports
the same C ABI (include/b200nb.h).  This module points the ctypes loader at that library and runs the parity cases of
tests/test_parity_gpu.py / tests/test_golden.py (the -m gpu tests) at reduced gene counts, with the same acceptance
rules.  What it buys: kernel control flow, indexing, shared-memory layout, warp synchronisation (the emulator does
not run lanes in lock step and reports collectives that not every named lane reaches) and use of uninitialised
memory (poisoned) are checked on every CPU run, before any GPU time is spent.  What it does not: performance, and
bit-identity with the GPU's arithmetic (tolerances are those of the GPU tests).

This is a CHECK of the product source, never a product path: the emulated library exists only under tests/, and
only this module (or an explicit B200NB_LIB=... in the environment of a test run, see DESIGN.md section 3.1) loads it.
The whole -m gpu suite (parity, golden files, device-resident pipeline, R shim, size factors, outlier refit) runs the
same way on a machine without a GPU, at the GPU tests' full sizes, the 50 000 x 100 config-2 case included (about
7 minutes; tests/helpers.py switches the torch tensors to the CPU when B200NB_LIB names the emulated library):

    B200NB_LIB=tests/simt_emu/_build/libb200nb_emu.so python -m pytest tests -m gpu
"""
import ctypes as C
import glob
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "simt_emu"))


def test_emulated_library_exports_the_c_abi(emu):
    from deseq2_b200 import _lib
    lib = _lib.lib()
    assert lib.b200nb_version().startswith(b"b200nb") and lib.b200nb_device_count() == 1
    before = lib.simt_emu_launches()
    x = np.array([0.3, 1.0, 7.5, 123.0])
    lg, dg, tg = np.empty(4), np.empty(4), np.empty(4)
    assert lib.b200nb_test_special(x.ctypes.data, 4, lg.ctypes.data, dg.ctypes.data, tg.ctypes.data) == 0
    assert lib.simt_emu_launches() > before            # the kernels really ran inside the emulator


import test_golden as TG          # noqa: E402
import test_parity_gpu as TP
import test_parity_reference_gpu as TPR      # noqa: E402
from reference_outputs import Reference  # noqa: E402


def _ref(case):
    return Reference("emulated_kernels", case)


CASES = [
    ("special functions", lambda e, o: TP.test_device_special_functions(e)),
    ("fitDisp MLE 800x37", lambda e, o: TP.test_fit_disp_mle_parity(e, o, 800, 37, 13)),
    ("fitDisp MLE m=6", lambda e, o: TP.test_fit_disp_mle_parity(e, o, 300, 6, 12)),
    ("fitDisp MAP m=100", lambda e, o: TP.test_fit_disp_map_parity(e, o, n=400)),
    ("fitDisp f64 counts, no CR", lambda e, o: TP.test_fit_disp_f64_counts_and_no_cr(e, o)),
    ("fitDisp TAB/BIG/GEN modes", lambda e, o: TP.test_fit_disp_big_and_mixed_counts(e, o, n=360)),
    ("fitDisp non-integer counts", lambda e, o: TP.test_fit_disp_non_integer_counts(e, o)),
    ("fitDisp weights ~condition", lambda e, o: TP.test_fit_disp_weights_and_designs(e, o, "condition", 51)),
    ("fitDisp weights ~batch+condition", lambda e, o: TP.test_fit_disp_weights_and_designs(e, o, "batch", 52)),
    ("fitDisp weights 4-level factor", lambda e, o: TP.test_fit_disp_weights_and_designs(e, o, "factor4", 53)),
    ("fitDisp CR column drop", lambda e, o: TP.test_fit_disp_weights_drop_a_design_column(e, o)),
    ("fitDispGrid", lambda e, o: TP.test_fit_disp_grid_parity(e, o)),
    ("fitBeta QR m=6", lambda e, o: TP.test_fit_beta_parity(e, o, 1500, 6, 32, True)),
    ("fitBeta normal equations m=37", lambda e, o: TP.test_fit_beta_parity(e, o, 800, 37, 33, False)),
    ("fitBeta maxit=0 contrast", lambda e, o: TP.test_fit_beta_maxit0_contrast(e, o)),
    ("fitBeta ~batch+condition, weights, nf matrix", lambda e, o: TP.test_fit_beta_designs_weights_nf_matrix(e, o, "batch", 61, True)),
    ("fitBeta 4-level factor", lambda e, o: TP.test_fit_beta_designs_weights_nf_matrix(e, o, "factor4", 62, False)),
    ("fitBeta intercept only", lambda e, o: TP.test_fit_beta_designs_weights_nf_matrix(e, o, "intercept", 63, True)),
    ("fitBeta badly scaled covariate", lambda e, o: TP.test_fit_beta_badly_scaled_covariate(e, o)),
    ("fitBeta divergence sentinel", lambda e, o: TP.test_fit_beta_divergence_sentinel(e)),
    ("fitBeta weight 0 == dropped sample", lambda e, o: TP.test_fit_beta_weight_zero_equals_dropped_sample(e)),
    ("general p: 10-level factor", lambda e, o: TP.test_general_p_parity(e, o, "factor10", 81, n=60)),
    ("general p: expanded 11 columns + ridge", lambda e, o: TP.test_general_p_parity(e, o, "expanded11", 82, n=60)),
    ("general p: continuous covariates", lambda e, o: TP.test_general_p_parity(e, o, "covariates7", 83, n=60)),
    ("segmented general p: m=7, 6 groups (saturated)", lambda e, o: TP.test_segmented_general_p_kernels(e, o, 7, 6, 1)),
    ("segmented general p: m=33, 6 groups", lambda e, o: TP.test_segmented_general_p_kernels(e, o, 33, 6, 3)),
    ("segmented general p: m=64, 12 groups", lambda e, o: TP.test_segmented_general_p_kernels(e, o, 64, 12, 4)),
    ("segmented general p: m=40, 32 groups", lambda e, o: TP.test_segmented_general_p_kernels(e, o, 40, 32, 7)),
    ("config 4 shape m=1000", lambda e, o: TP.test_config_shapes_spot_check(e, o, "C4", 48, 1000)),
    ("config 3 shape m=500", lambda e, o: TP.test_config_shapes_spot_check(e, o, "C3", 60, 500)),
    ("edge 1x4", lambda e, o: TP.test_edge_shapes(e, o, 1, 4)),
    ("edge 3x5", lambda e, o: TP.test_edge_shapes(e, o, 3, 5)),
    ("edge 7x33", lambda e, o: TP.test_edge_shapes(e, o, 7, 33)),
    ("edge 2x3000", lambda e, o: TP.test_edge_shapes(e, o, 2, 3000)),
    ("empty input", lambda e, o: TP.test_empty_input_is_a_no_op(e)),
    ("engine vs the reference TU: fitDisp m=24", lambda e, o: TPR.test_fit_disp_vs_reference(e, o, _ref("fitDisp m=24"), 300, 24, 213)),
    ("engine vs the reference TU: fitBeta m=6", lambda e, o: TPR.test_fit_beta_vs_reference(e, _ref("fitBeta m=6"), 300, 6, 222, True)),
    ("engine vs the reference TU: general p, weights, ridge", lambda e, o: TPR.test_fit_beta_weights_ridge_general_p_vs_reference(e, _ref("general p"))),
    ("host input cache: content-addressed, never stale", lambda e, o: TP.test_host_cache_is_content_addressed_and_never_stale(e, o)),
    ("post-rule parity m=4 (Monte-Carlo prior variance)", lambda e, o: TP.test_post_rule_parity_every_gene(e, o, 4, 250, 0.3)),
    ("post-rule parity m=6", lambda e, o: TP.test_post_rule_parity_every_gene(e, o, 6, 300, 0.25)),
    ("post-rule parity m=12", lambda e, o: TP.test_post_rule_parity_every_gene(e, o, 12, 250, 0.12)),
]


@pytest.mark.parametrize("name,run", CASES, ids=[c[0] for c in CASES])
def test_emulated_kernel_parity(emu, oracle, name, run):
    run(emu, oracle)


@pytest.fixture()
def emu_device(emu, monkeypatch):
    """deseq2_b200.device / device_pipeline on CPU torch tensors: in the emulator "device" pointers are host pointers
    and there are no streams, so the torch plumbing runs unchanged with device = "cpu"."""
    import test_device_pipeline_gpu as TD
    from deseq2_b200 import device as D, device_pipeline as DP
    null_stream = lambda: C.c_void_p(0)
    monkeypatch.setattr(D, "_stream", null_stream)
    monkeypatch.setattr(DP, "_stream", null_stream)
    monkeypatch.setattr(TD, "DEV", "cpu")
    import test_size_factors_gpu as TS
    monkeypatch.setattr(TS, "DEV", "cpu")
    TD.TS = TS
    DP._ws.clear() if hasattr(DP._ws, "clear") else None
    return TD


DEVICE_CASES = [
    ("prep ~condition", lambda T, e: T.test_prep_kernel_matches_numpy(e, "condition", n=300)),
    ("prep ~batch+condition", lambda T, e: T.test_prep_kernel_matches_numpy(e, "batch", n=300)),
    ("prep per group: ~batch+condition m=300", lambda T, e: T.test_prep_kernel_matches_numpy(e, "batch-long-rows", n=120)),
    ("prep per group: 10-level factor m=300", lambda T, e: T.test_prep_kernel_matches_numpy(e, "factor10-long-rows", n=120)),
    ("prep streaming: covariates m=300", lambda T, e: T.test_prep_kernel_matches_numpy(e, "covariates-long-rows", n=120)),
    ("trend fit", lambda T, e: T.test_trend_kernel_matches_numpy(e, n=3000)),
    ("cooks m=12", lambda T, e: T.test_cooks_kernel_matches_numpy(e, "condition", 12, n=200)),
    ("cooks ~batch+condition", lambda T, e: T.test_cooks_kernel_matches_numpy(e, "batch", 36, n=150)),
    ("cooks covariate (one cell per sample)", lambda T, e: T.test_cooks_kernel_matches_numpy(e, "covariate", 20, n=150)),
    ("cooks 10-level factor", lambda T, e: T.test_cooks_kernel_matches_numpy(e, "factor10", 200, n=60)),
    ("cooks cells of 75 (4 entries per lane)", lambda T, e: T.test_cooks_kernel_matches_numpy(e, "condition", 150, n=40)),
    ("cooks cells of 200 (8 entries per lane)", lambda T, e: T.test_cooks_kernel_matches_numpy(e, "condition", 400, n=30)),
    ("cooks cells of 350 (extraction path)", lambda T, e: T.test_cooks_kernel_matches_numpy(e, "condition", 700, n=20)),
    ("cooks covariate m=100 (one cell per sample)", lambda T, e: T.test_cooks_kernel_matches_numpy(e, "covariate", 100, n=40)),
    ("DESeq on device ~condition", lambda T, e, o: T.test_device_pipeline_matches_host_pipeline(e, o, "condition", 240, 40)),
    ("DESeq on device ~condition m=6", lambda T, e, o: T.test_device_pipeline_matches_host_pipeline(e, o, "condition", 300, 6)),
    ("DESeq on device ~batch+condition", lambda T, e, o: T.test_device_pipeline_matches_host_pipeline(e, o, "batch", 160, 36)),
    ("long rows (m >= 400) on the segmented kernels", lambda T, e, o: T.test_long_rows_take_the_segmented_kernels(e, o)),
    ("LRT on device", lambda T, e: T.test_lrt_device_matches_host(e, n=250)),
    ("optim fallback on device", lambda T, e: T.test_optim_fallback_device_vs_host(e, n=120)),
    ("size factors 700x12", lambda T, e: T.TS.test_size_factors_match_numpy(e, 700, 12, 1, False)),
    ("size factors 501x37 double", lambda T, e: T.TS.test_size_factors_match_numpy(e, 501, 37, 2, True)),
    ("size factors 150x130", lambda T, e: T.TS.test_size_factors_match_numpy(e, 150, 130, 3, False)),
    ("size factors 64x5", lambda T, e: T.TS.test_size_factors_match_numpy(e, 64, 5, 4, False)),
    ("size factors degenerate", lambda T, e: T.TS.test_size_factors_degenerate_inputs(e)),
    ("DESeq on device from raw counts", lambda T, e: T.TS.test_deseq_device_from_raw_counts(e, n=200)),
    ("outlier replacement + refit ~condition", lambda T, e: T.TS.test_outlier_replacement_and_refit_device_vs_host(e, "condition", n=300)),
    ("getContrast on device", lambda T, e: T.TS.test_get_contrast_device_matches_host(e, n=200)),
    ("outlier replacement + refit, mixed cells", lambda T, e: T.TS.test_outlier_replacement_and_refit_device_vs_host(e, "mixed", n=300)),
]


@pytest.mark.parametrize("name,run", DEVICE_CASES, ids=[c[0] for c in DEVICE_CASES])
def test_emulated_device_pipeline(emu, emu_device, oracle, name, run):
    import inspect
    if len(inspect.signature(run).parameters) == 3:
        run(emu_device, emu, oracle)
    else:
        run(emu_device, emu)


def test_emulated_engine_through_R_boundary(emu, oracle, tmp_path):
    """The R .Call shim linked against the emulated engine: R-shaped arguments in, the CUDA kernels' source executed,
    named R list out -- the complete drop-in path of INTEGRATION.md, minus R and minus the GPU."""
    import build_emu
    import test_r_shim as TR
    path = build_emu.build()
    so = TR._build(str(tmp_path), "DESeq2_emu.so", [], [path, "-Wl,-rpath," + os.path.dirname(path)])
    TR.test_engine_through_R_boundary(TR.MockR(so), oracle)


_CHUNK_PROBE = r"""
import sys
import numpy as np
sys.path.insert(0, {root!r}); sys.path.insert(0, {tests!r})
from deseq2_b200 import wrappers as W
from helpers import make_case, disp_args, beta_args
c = make_case(500, 37, seed=5)
g = W.fitDisp(**disp_args(c, c["mu"], np.log(c["alpha0"])))
alpha = np.exp(g["log_alpha"])
w = np.random.default_rng(1).uniform(0.3, 1, c["counts"].shape)
b = W.fitBeta(**beta_args(c, alpha, weights=w, useWeights=True), return_mu=True)
grid = np.linspace(np.log(1e-8), np.log(30), 20)
gg = W.fitDispGrid(ySEXP=c["counts"].astype(np.float64), xSEXP=c["x"], mu_hatSEXP=c["mu"], disp_gridSEXP=grid,
                   log_alpha_prior_meanSEXP=np.log(alpha), log_alpha_prior_sigmasqSEXP=0.5, usePriorSEXP=True,
                   weightsSEXP=w, useWeightsSEXP=True, weightThresholdSEXP=1e-2, useCRSEXP=True)
out = dict(grid=gg["log_alpha"])
out.update(("d_" + k, v) for k, v in g.items())
out.update(("b_" + k, v) for k, v in b.items())
np.savez(sys.argv[1], **out)
"""


def test_chunked_host_path_is_bit_identical(emu, tmp_path):
    """B200NB_CHUNK_GENES (capi.cu run_chunked: gene blocks of the R-layout arrays handled by worker threads with their
    own streams / workspaces / pinned rings) must return exactly what the unchunked call returns: strided gather of
    the column-major inputs, per-block launches, strided scatter of hat_diagonals / mu / beta matrices."""
    import subprocess
    import build_emu
    script = tmp_path / "probe.py"
    script.write_text(_CHUNK_PROBE.format(root=os.path.dirname(HERE), tests=HERE))
    outs = {}
    for tag, extra in (("whole", {}), ("w1", {"B200NB_CHUNK_GENES": "97", "B200NB_CHUNK_WORKERS": "1"}),
                       ("w3", {"B200NB_CHUNK_GENES": "61", "B200NB_CHUNK_WORKERS": "3"})):
        env = dict(os.environ, B200NB_LIB=build_emu.build(), **extra)
        env.pop("B200NB_FORCE_GENERIC", None)
        f = str(tmp_path / (tag + ".npz"))
        r = subprocess.run([sys.executable, str(script), f], env=env, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        outs[tag] = np.load(f)
    assert len(outs["whole"].files) == 18
    for tag in ("w1", "w3"):
        for k in outs["whole"].files:
            assert np.array_equal(outs["whole"][k], outs[tag][k], equal_nan=True), (tag, k)


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(HERE, "golden", "*.npz"))), ids=os.path.basename)
def test_emulated_engine_matches_golden(emu, path):
    TG.test_engine_matches_golden(emu, path)


@pytest.mark.parametrize("lanes", [8, 16, 32])
def test_every_group_width_keeps_parity(lanes):
    """The small-p kernels run one, two or four genes per warp (32 / 16 / 8 lanes per gene; chosen from the number of
    samples at run time, B200NB_GROUP_LANES forces one).  Whatever the width, results must be the oracle's: a slice of
    the parity suite with each width forced, in a fresh process (the choice is read once per process)."""
    import subprocess
    import build_emu
    lib = build_emu.build()
    sel = "800-37 or 1500-6 or big_and_mixed or maxit0 or condition-51 or batch-61 or edge_shapes or divergence"
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.join(HERE, "test_parity_gpu.py"), "-q", "-m", "gpu", "-x",
                        "-p", "no:cacheprovider", "-k", sel],
                       env=dict(os.environ, B200NB_LIB=lib, B200NB_GROUP_LANES=str(lanes)), capture_output=True,
                       text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-1000:]
    assert " passed" in r.stdout and "failed" not in r.stdout


def test_microbench_program_runs_against_the_emulated_engine(emu, tmp_path):
    """scripts/microbench.cu (the Python-free A/B timer for the GPU box) compiled against the emulator's runtime header:
    device mode on two libraries (the second must reproduce the first to rounding) and host mode with the chunked path."""
    import subprocess
    import build_emu
    exe = str(tmp_path / "microbench_emu")
    sim = os.path.join(HERE, "simt_emu")
    subprocess.run(["/usr/bin/g++", "-std=c++17", "-O1", "-x", "c++", "-w", "-I", sim, "-o", exe,
                    os.path.join(os.path.dirname(HERE), "scripts", "microbench.cu"), os.path.join(sim, "emu.cpp"), "-ldl"],
                   check=True, capture_output=True, text=True)
    lib = build_emu.build()
    env = dict(os.environ, B200NB_TEST_EMULATOR="1")
    r = subprocess.run([exe, "--genes", "150", "--samples", "24", "--reps", "1", lib, lib], env=env, capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = [l for l in r.stdout.splitlines() if "fitDisp" in l and "fitBeta" in l]
    assert len(lines) == 2 and "max|dlog_alpha| 0.00e+00" in lines[1] and "max|dbeta| 0.00e+00" in lines[1]
    r = subprocess.run([exe, "--host", "--genes", "150", "--samples", "24", "--reps", "1", lib],
                       env=dict(env, B200NB_CHUNKS="3"), capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "end to end" in r.stdout, r.stdout + r.stderr
