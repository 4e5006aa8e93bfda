#!/usr/bin/env python
"""bench.py -- genes/sec of the DESeq2 Wald hot path (fitDisp MLE + fitDisp MAP + fitBeta) on B200.

Contract (see task text): `python bench.py --gpus N --steps K --warmup W` prints ONE JSON line on rank 0.
  step      one pass of the hot path over one batch of synthetic counts: fitDisp (gene-wise MLE) ->
            fitDisp (MAP, prior from the fitted trend) -> fitBeta (Wald IRLS), the three native calls of
            DESeq()'s default Wald path for a linear-mu design (SURVEY.md 8d).
  value     genes/sec, kernels only, inputs resident in HBM (gene-major), CUDA events, max over ranks.
  e2e       the same three calls through the C ABI with HOST buffers in R layout (b200nb_fit_disp x2,
            b200nb_fit_beta): H2D, layout conversion, kernels, D2H all inside the timed region.
  roofline  dominant kernel = fit_disp (MLE launch): algorithmic bytes n*(12m+88) / CUDA-event time vs the
            measured HBM copy bandwidth (MEASURED_PEAKS.json).  The path is FP64-pipe bound (DESIGN.md), so
            the HBM fraction is small by construction; it is reported because the contract asks for it.
  cpu_baseline / --impl reference: the oracle (C restatement of src/DESeq2.cpp, all host threads) on a
            bounded sample of the same workload.  R is not in this image, so kind = "port".
N > 1: every rank owns its own shard of n genes (weak scaling); per step the per-gene results
(beta, SE, dispersion) are all-gathered over NCCL so rank 0 holds them (R/parallel.R:54-66's rbind).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MIN_LOG_ALPHA = float(np.log(1e-8 / 10))


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--genes", type=int, default=50000, help="genes per GPU (config C2: 50k)")
    ap.add_argument("--samples", type=int, default=100)
    ap.add_argument("--cpu-sample", type=int, default=20000, help="genes in the CPU baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the BASELINE configs 3-5 block")
    ap.add_argument("--quick-configs", action="store_true", help="configs block at 20%% of the stated sizes")
    ap.add_argument("--r-default-probe", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (float64; a fixed, seeded "
                         "sample of the genes of large outputs), so two builds can be compared output for output; "
                         "with more than one GPU: rank 0's own shard, not the gathered results")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


# ---------------------------------------------------------------- workload

def build_workload(n, m, seed, engine):
    """Synthetic C2 workload + the exact inputs of the three native calls, produced by one untimed run of the
    host pipeline with `engine` (so MAP/fitBeta inputs are the real downstream values)."""
    from deseq2_b200 import pipeline, synth
    d = synth.make_example_counts(n, m, seed=seed)
    counts = d["counts"]
    counts = counts[counts.sum(axis=1) > 0]
    x, sf = d["x"], d["sizeFactors"]
    ge = pipeline.estimateDispersionsGeneEst(counts, sf, x, engine=engine)
    tf = pipeline.estimateDispersionsFit(ge["dispGeneEst"], ge["baseMean"])
    pv = pipeline.estimateDispersionsPriorVar(tf["varLogDispEsts"], m, x.shape[1], ge["dispGeneEst"], tf["dispFit"])
    mp = pipeline.estimateDispersionsMAP(counts, x, ge["mu"], ge["dispGeneEst"], tf["dispFit"], pv,
                                         tf["varLogDispEsts"], engine=engine)
    norm = counts / sf[None, :]
    rough = pipeline.roughDispEstimate(norm, x)
    mom = pipeline.momentsDispEstimate(ge["baseMean"], ge["baseVar"], sf)
    alpha0 = np.minimum(np.maximum(1e-8, np.minimum(rough, mom)), max(10, m))
    dispInit = np.where(ge["dispGeneEst"] > 0.1 * tf["dispFit"], ge["dispGeneEst"], tf["dispFit"])
    Q, R = np.linalg.qr(x)
    beta0 = np.linalg.solve(R, Q.T @ np.log(norm + 0.1).T).T
    # host buffers in R layout (column-major), exactly what .Call would hand over: no conversion in the timed region
    F = np.asfortranarray
    nf = F(np.broadcast_to(sf[None, :], counts.shape).astype(np.float64))
    return dict(counts=F(counts), x=F(x), sf=sf, nf=nf, mu=F(ge["mu"]), log_alpha0=np.log(alpha0),
                log_dispInit=np.log(dispInit), log_dispFit=np.log(tf["dispFit"]), priorVar=pv,
                dispersion=mp["dispersion"], beta0=F(beta0), lam=np.full(x.shape[1], 1e-6) / np.log(2) ** 2)


def three_calls_host(w, engine, sl=slice(None)):
    """The hot path through the reference-facing API with host buffers (argument names of src/DESeq2.cpp)."""
    c, x, mu = w["counts"][sl], w["x"], w["mu"][sl]
    n, m = c.shape
    common = dict(ySEXP=c, xSEXP=x, mu_hatSEXP=mu, min_log_alphaSEXP=MIN_LOG_ALPHA, kappa_0SEXP=1.0, tolSEXP=1e-6,
                  maxitSEXP=100, weightsSEXP=None, useWeightsSEXP=False, weightThresholdSEXP=1e-2, useCRSEXP=True)
    r1 = engine.fitDisp(log_alphaSEXP=w["log_alpha0"][sl], log_alpha_prior_meanSEXP=w["log_alpha0"][sl],
                        log_alpha_prior_sigmasqSEXP=1.0, usePriorSEXP=False, **common)
    r2 = engine.fitDisp(log_alphaSEXP=w["log_dispInit"][sl], log_alpha_prior_meanSEXP=w["log_dispFit"][sl],
                        log_alpha_prior_sigmasqSEXP=w["priorVar"], usePriorSEXP=True, **common)
    r3 = engine.fitBeta(ySEXP=c, xSEXP=x, nfSEXP=w["nf"][sl], alpha_hatSEXP=w["dispersion"][sl],
                        contrastSEXP=np.r_[1.0, np.zeros(x.shape[1] - 1)], beta_matSEXP=w["beta0"][sl],
                        lambdaSEXP=w["lam"], weightsSEXP=None, useWeightsSEXP=False, tolSEXP=1e-8, maxitSEXP=100,
                        useQRSEXP=True, minmuSEXP=0.5)
    return r1, r2, r3


def host_bytes(n, m, p):
    h2d = 2 * (4 * n * m + 8 * n * m + 16 * n + 8 * m * p) + (4 * n * m + 8 * n * m + 8 * n + 8 * n * p + 8 * m * p + 16 * p)
    d2h = 2 * (7 * 8 * n + 2 * 4 * n) + (8 * n * m + 2 * 8 * n * p + 4 * 8 * n)
    return h2d, d2h


# ---------------------------------------------------------------- clocks

class ClockSampler:
    """SM clock / throttle-reason log for the timed region, the way /opt/skills/guides/B200_PROFILING.md does it: a
    separate `nvidia-smi -lms` process started BEFORE the warm-up and stopped after the run (in-process NVML polling
    was measured to stall the launching thread by 0.3-3 ms per query; a forked nvidia-smi per sample by far more).
    Rows are attributed to the timed region by their timestamps; the GPU is kept under the same load until at least
    two rows fall inside [start of timed region, now]."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index, period_ms=200):
        self.index, self.period_ms = index, period_ms
        self.proc, self.window, self._buf, self._t = None, None, [], None

    def start(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = vis.split(",")[self.index] if vis else str(self.index)
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms",
                                          str(self.period_ms), "-i", phys], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True, bufsize=1)
            self._t = threading.Thread(target=self._reader, daemon=True)
            self._t.start()
            # nvidia-smi's own start-up (NVML init over every GPU of the box) holds driver locks for 100s of ms and was
            # measured to stall our kernels: wait for its first row before any timed work is enqueued
            t0 = time.time()
            while not self._buf and time.time() - t0 < 10.0 and self.proc.poll() is None:
                time.sleep(0.01)
        except Exception:
            self.proc = None

    def _reader(self):
        for line in self.proc.stdout:
            self._buf.append((time.time(), line))

    def rows_since(self, t0):
        return [r for r in self._buf if r[0] >= t0]

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "source": "unavailable"}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=3)
        except Exception:
            self.proc.kill()
        rows = self._buf
        if self.window is not None:
            inside = [r for r in rows if self.window[0] <= r[0] <= self.window[1]]
            rows = inside if inside else rows[-2:]
        sm, mx, reasons = [], [], set()
        for _, line in rows:
            f = [v.strip() for v in line.split(",")]
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except Exception:
                continue
            for k, nm in enumerate(self.NAMES):
                if len(f) > 3 + k and f[3 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm),
                "source": f"nvidia-smi -lms {self.period_ms}, rows from the start of the timed region while the same steps keep running"}


# ---------------------------------------------------------------- reference arm / cpu baseline

def host_threads():
    """CPU threads this process may actually use: the affinity mask, capped by a cgroup CPU quota when there is one
    (os.cpu_count() reports the whole machine even inside a 1-GPU lease; round 1's CPU arm swung 6x between two boxes
    because it asked for 128 threads regardless)."""
    n = len(os.sched_getaffinity(0))
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period))))
    except Exception:
        pass
    return int(os.environ.get("B200NB_REF_THREADS", n))


def limit_library_thread_pools():
    """numpy's OpenBLAS and torch's OpenMP pool start one worker per CPU of the affinity mask (64-128 on the GPU
    hosts) and those workers busy-wait after every call; inside a container with a CPU quota (1-GPU lease: 16 CPUs) the
    spin exhausts the quota and the kernel throttles the whole process for the rest of the 100 ms period -- holes of
    40-90 ms in a device pipeline whose host glue is a few numpy calls (profiles/r02_pipeline_host_stalls.md).  The GPU
    arm needs none of those pools: one thread each.  (torchrun does the same with OMP_NUM_THREADS=1 for N > 1.)"""
    done = []
    try:
        import threadpoolctl
        threadpoolctl.threadpool_limits(1)
        done.append("threadpoolctl: 1")
    except Exception:
        pass
    try:
        import torch
        torch.set_num_threads(1)
        done.append("torch: 1")
    except Exception:
        pass
    return ", ".join(done) or "unchanged"


class RefEngine:
    """The CPU arm's engine: the REFERENCE'S OWN src/DESeq2.cpp (oracle/_ref, compiled unchanged against stand-in
    headers; kind = "reference") with `threads` BiocParallel-style gene chunks (R/parallel.R:9-10); if the prebuilt
    library is missing (it is built in the build container only) the oracle restatement (kind = "port")."""

    def __init__(self, threads):
        from oracle import ref as R
        self.threads = threads
        if R.available():
            R.build()
            R.lib()
            self.kind, self.R = "reference", R
            self.what = "/root/reference/src/DESeq2.cpp compiled unchanged (oracle/_ref, stand-in Rcpp/Armadillo/Rmath headers)"
        else:
            from oracle import oracle as O
            import ctypes
            O.build()
            O.lib()
            try:
                ctypes.CDLL("libgomp.so.1").omp_set_num_threads(int(threads))
            except Exception:
                pass
            self.kind, self.R = "port", O
            self.what = "oracle C restatement of src/DESeq2.cpp (oracle/_ref not available on this box)"

    def _kw(self):
        return {"nthreads": self.threads} if self.kind == "reference" else {}

    def fitDisp(self, **kw):
        return self.R.fitDisp(**kw, **self._kw())

    def fitDispGrid(self, **kw):
        return self.R.fitDispGrid(**kw, **self._kw())

    def fitBeta(self, **kw):
        return self.R.fitBeta(**kw, **self._kw())


def time_reference(w, n_sample, steps, warmup, threads, budget_s=100.0):
    """The three calls of one step on the first n genes of the workload with `threads` host threads.  The sample is
    shrunk if the requested steps would not fit the time budget.  Returns (genes/s, s per step, n, engine)."""
    eng = RefEngine(threads)
    n = min(n_sample, len(w["counts"]))
    probe = min(n, max(200, 40 * threads))
    three_calls_host(w, eng, slice(0, probe))                # thread start-up, first touch of the workspaces
    t0 = time.perf_counter()
    three_calls_host(w, eng, slice(0, probe))
    per_gene = (time.perf_counter() - t0) / probe
    total_passes = max(1, steps + warmup)
    if per_gene * n * total_passes > budget_s:
        n = max(probe, int(budget_s / (per_gene * total_passes)))
    sl = slice(0, n)
    for _ in range(warmup):
        three_calls_host(w, eng, sl)
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        three_calls_host(w, eng, sl)
        ts.append(time.perf_counter() - t0)
    dt = float(np.median(ts))
    return n / dt, dt, n, eng


def cpu_baseline_record(w, n_sample, steps, warmup):
    """cpu_baseline of the bench line: the reference on all usable host threads (value) and on one thread (the
    reference's own default, parallel = FALSE, R/core.R:287)."""
    T = host_threads()
    v, dt, ns, eng = time_reference(w, n_sample, steps, warmup, T)
    v1, dt1, ns1, _ = time_reference(w, min(n_sample, 1500), 1, 0, 1, budget_s=20.0)
    return {"value": v, "unit": "genes/s", "cores": T, "kind": eng.kind,
            "sample": f"first {ns} genes of the workload (fitDisp MLE + fitDisp MAP + fitBeta), {eng.what}, {T} threads "
                      f"= contiguous gene chunks (BiocParallel emulation), median of {steps} passes of {dt:.2f} s",
            "single_thread": {"value": v1, "unit": "genes/s", "cores": 1,
                              "sample": f"first {ns1} genes, one pass of {dt1:.2f} s (the reference's default parallel=FALSE)"}}


def r_default_probe(n, m):
    """Child-process mode of the GPU arm: the device-resident DESeq() with R's defaults (size factors from the raw counts,
    outlier replacement + refit) on the C2 workload; prints one JSON object."""
    import torch
    from deseq2_b200 import device as D, device_pipeline as DP, synth
    d = synth.make_example_counts(n, m, seed=20260923 + 2)
    counts = d["counts"][d["counts"].sum(axis=1) > 0]
    y = D.to_gene_major(np.ascontiguousarray(counts), torch.device("cuda", 0))
    for _ in range(2):
        DP.DESeq_device(y, d["x"], None, minReplicatesForReplace=7)
    torch.cuda.synchronize()
    ts = []
    for _ in range(5):
        t0 = time.perf_counter()
        rr = DP.DESeq_device(y, d["x"], None, minReplicatesForReplace=7)
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    dt = float(np.median(ts))
    print(json.dumps({"value": len(counts) / dt, "unit": "genes/s (one GPU)", "ms_per_step": dt * 1e3,
                      "genes_refitted": int(rr.get("n_replaced", 0)),
                      "what": "size factors on device + full_pipeline + outlier replacement and refit"}))


def bind_to_gpu_numa_node(torch, local_rank):
    """One process per GPU: run this rank (and so first-touch its host buffers, its pinned staging ring and its result
    arrays) on the CPUs of the NUMA node the GPU hangs off -- what `numactl --cpunodebind` does for an R worker per
    GPU.  torchrun starts the ranks unpinned; round 1's e2e fell to 0.475 efficiency at 8 GPUs with every rank staging
    through whichever socket it happened to run on.  B200NB_BENCH_NUMA=0 switches it off."""
    if os.environ.get("B200NB_BENCH_NUMA", "1") == "0":
        return "off"
    try:
        pr = torch.cuda.get_device_properties(local_rank)
        bus = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return "unknown node"
        cpus = set()
        for tok in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = tok.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return "no usable cpu on node %d" % node
        os.sched_setaffinity(0, cpus)
        return "rank bound to NUMA node %d (%d CPUs)" % (node, len(cpus))
    except Exception as ex:  # pragma: no cover
        return "not bound: " + repr(ex)[:80]


def configs_block(world, rank, dev, peak_gbs, quick=False):
    """BASELINE.json configs 3, 4, 5 through the device-resident pipeline (deseq2_b200.device_pipeline / sharded): the
    whole DESeq() sequence of each config -- pre-steps, fitBeta for the GeneEst means where the design is not
    group-wise (C3, C5), both dispersion fits, trend, grid refits, the Wald / LRT fits, Cook's -- with the counts
    resident in HBM, timed with CUDA events (max over ranks), incl. the pipeline's few host syncs.
      N = 1: C4 at its stated size (50k x 1000, 10-level factor) and C3 / C5 at their per-GPU shard size on 8 GPUs.
      N > 1: C3 (200k x 500) and C5 (1M x 200, LRT) at their stated TOTAL size, gene-sharded over the N ranks with one
             packed all-gather for the global step and ONE packed all-gather of the results (sharded.PackedGather),
             plus C2 strong scaling (the 50k genes of config 2 split over the ranks, kernels only).
    Algorithmic bytes per gene are SURVEY.md section 8(d)'s."""
    import torch
    import torch.distributed as dist
    from deseq2_b200 import device as D, device_pipeline as DP, sharded, synth
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def timed(fn, reps=3):
        r = fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            if world > 1:
                dist.barrier()
            a_, b_ = ev(), ev()
            a_.record()
            r = fn()
            b_.record()
            torch.cuda.synchronize()
            t = torch.tensor([a_.elapsed_time(b_)], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ts.append(float(t.item()))
        return float(np.median(ts)), r

    def total(v):
        t = torch.tensor([float(v)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    def common_sf(m, seed):     # the experiment's size factors: the same on every rank
        sf = np.exp(np.random.Generator(np.random.PCG64(seed)).normal(0.0, 0.25, m))
        return sf / np.exp(np.mean(np.log(sf)))

    def shard(n_total, m, x, seed, **kw):
        lo, hi = sharded.shard_bounds(n_total, world, rank)
        sf = common_sf(m, seed)
        d = synth.make_example_counts(hi - lo, m, x=x, seed=seed + 17 * (rank + 1), sizeFactors=sf, **kw)
        return D.to_gene_major(d["counts"], dev), sf

    out = {}
    scale = 0.2 if quick else 1.0
    specs = []
    if world == 1:
        specs.append(("C4", int(50000 * scale), 1000, synth.design_factor(1000, 10), "wald", 64 * 1000 + 24 * 21 + 256))
        specs.append(("C3_shard_of_8", int(25000 * scale), 500, synth.design_batch_condition(500, 3), "wald", 64 * 500 + 48 * 4 + 256))
        specs.append(("C5_shard_of_8", int(125000 * scale), 200, synth.design_batch_condition(200, 2), "lrt", 84 * 200 + 24 * 8 + 296))
    else:
        specs.append(("C3", int(200000 * scale), 500, synth.design_batch_condition(500, 3), "wald", 64 * 500 + 48 * 4 + 256))
        specs.append(("C5", int(1000000 * scale), 200, synth.design_batch_condition(200, 2), "lrt", 84 * 200 + 24 * 8 + 296))
    for name, n_total, m, x, kind, bytes_per_gene in specs:
        try:
            y, sf = shard(n_total, m, x, 20260923 + len(name), betaSD=0.5)
            p = x.shape[1]
            if world > 1:
                run = lambda: sharded.sharded_DESeq_device(y, x, sf)
            else:
                run = lambda: DP.DESeq_device(y, x, sf)
            ms, res = timed(run)
            genes = total(res["idx"].numel())
            rec = {"genes_total": int(genes), "genes_per_rank": int(y.shape[0]), "samples": m, "p": p, "n_gpus": world,
                   "deseq_device_ms": ms, "genes_per_s": genes / (ms * 1e-3),
                   "alg_bytes_per_gene": bytes_per_gene,
                   "hbm_frac": genes * bytes_per_gene / (ms * 1e-3) / 1e9 / peak_gbs,
                   "n_optim_rows": int(total(res.get("n_optim", 0)))}
            if world > 1:
                rec["per_gene_collectives"] = int(res["collectives"]) - 1
            if kind == "lrt":
                ynz = y[res["idx"]].contiguous()
                xr = x[:, :2]
                if world > 1:
                    lrt = lambda: sharded.sharded_nbinomLRT_device(ynz, x, xr, sf, res["dispersion"])
                else:
                    lrt = lambda: DP.nbinomLRT_device(ynz, x, xr, sf, res["dispersion"])
                ms2, _ = timed(lrt)
                rec["nbinomLRT_device_ms"] = ms2
                rec["genes_per_s_incl_lrt"] = genes / ((ms + ms2) * 1e-3)
            if world == 1:
                os.environ["B200NB_PIPE_DEBUG"] = "1"      # one extra run with a sync after every stage
                try:
                    rec["stage_ms"] = run()["stage_ms"]
                finally:
                    del os.environ["B200NB_PIPE_DEBUG"]
                hot = [rec["stage_ms"].get(k) for k in ("fit_disp_mle", "fit_disp_map", "fit_beta")]
                if all(v is not None for v in hot):
                    # the three native calls of the Wald path inside this run (stage wall times with a sync after each)
                    rec["hot_path_ms"] = round(sum(hot), 3)
                    rec["hot_path_genes_per_s"] = genes / (sum(hot) * 1e-3)
            out[name] = rec
            del y, res
            torch.cuda.empty_cache()
        except Exception as ex:  # pragma: no cover
            out[name] = {"error": repr(ex)[:300]}
    if world > 1:
        # strong scaling of config 2: its 50 000 genes split over the ranks, the three kernels, device resident
        try:
            n2, m2 = int(50000 * scale), 100
            x2 = synth.design_condition(m2)
            lo, hi = sharded.shard_bounds(n2, world, rank)
            sf2 = common_sf(m2, 20260925)
            d = synth.make_example_counts(hi - lo, m2, x=x2, seed=20260923 + 2 + rank, sizeFactors=sf2)
            y2 = D.to_gene_major(d["counts"], dev)
            pr = DP.prep(y2, x2, sf2)
            la0 = torch.log(pr["alpha0"])
            lam = torch.full((2,), 1e-6 / np.log(2) ** 2, dtype=torch.float64, device=dev)
            con = torch.tensor([1.0, 0.0], dtype=torch.float64, device=dev)

            def three():
                r1 = D.fit_disp(y2, pr["xd"], pr["mu_lin"], la0, la0, 1.0, MIN_LOG_ALPHA, 1.0, 1e-6, 100, False)
                r2 = D.fit_disp(y2, pr["xd"], pr["mu_lin"], r1["log_alpha"], la0, 1.0, MIN_LOG_ALPHA, 1.0, 1e-6, 100, True)
                return D.fit_beta(y2, pr["xd"], pr["sfd"], torch.exp(r2["log_alpha"]), con, pr["beta0"], lam, 1e-8, 100)
            ms, _ = timed(three, reps=5)
            out["C2_strong_scaling"] = {"genes_total": n2, "genes_per_rank": hi - lo, "n_gpus": world, "kernels_ms": ms,
                                        "genes_per_s": n2 / (ms * 1e-3),
                                        "what": "fitDisp + fitDisp(prior) + fitBeta on 1/N of config 2's genes per GPU, "
                                                "device resident, CUDA events, max over ranks"}
        except Exception as ex:  # pragma: no cover
            out["C2_strong_scaling"] = {"error": repr(ex)[:300]}
    return out


def last_step_outputs(outs, ng, m, max_genes=100000, matrix_bytes=32 << 20):
    """What the three calls of a step return to their caller, as float64 host arrays: fitDisp MLE and MAP
    (fitdisp_mle_*, fitdisp_map_*: the nine per-gene list members) and fitBeta (fitbeta_*: beta_mat and beta_var_mat
    as n x p, the per-gene vectors, hat_diagonals and mu as n x m).  Rows past ng only pad a shard.  A fixed, seeded
    sample of the genes is kept where there are more than max_genes, and of the n x m matrices as many rows as fit
    matrix_bytes; the row indices are stored as rows_vectors and rows_matrices.  The per-gene arrays take at most
    (23 + 2 p) * 8 * max_genes bytes (21.6 MB for the benchmark's p = 2) and the two matrices at most matrix_bytes
    (33.6 MB), so the dump stays below 64 MB for any number of genes and samples."""
    max_matrix_rows = min(4096, matrix_bytes // (2 * 8 * m))
    pick = lambda k: np.sort(np.random.default_rng(0).choice(ng, k, replace=False)) if k < ng else np.arange(ng)
    rv, rm = pick(max_genes), pick(max_matrix_rows)
    out = {"rows_vectors": rv.astype(np.float64), "rows_matrices": rm.astype(np.float64)}
    for prefix, d in (("fitdisp_mle_", outs[0]), ("fitdisp_map_", outs[1]), ("fitbeta_", outs[2])):
        for k, t in d.items():
            if t is None:
                continue
            v = t.detach().cpu().numpy().astype(np.float64)
            if k in ("beta_mat", "beta_var_mat"):
                out[prefix + k] = v.T[rv]
            elif v.ndim == 2:
                out[prefix + k] = v[rm, :m]
            else:
                out[prefix + k] = v[rv]
    return out


def main():
    a = parse()
    if a.r_default_probe:
        return r_default_probe(a.genes, a.samples)
    # NCCL's own log (version banner, communicator init lines with nranks) must not land on stdout, where the ONE JSON
    # line goes -- and must not be hidden either: it goes to stderr at INFO/INIT level unless the caller chose otherwise
    # (NCCL ignores NCCL_DEBUG_FILE at the VERSION level some images preset, and then prints its banner on stdout)
    if os.environ.get("NCCL_DEBUG", "").upper() not in ("INFO", "TRACE"):
        os.environ["NCCL_DEBUG"] = "INFO"
        os.environ.setdefault("NCCL_DEBUG_SUBSYS", "INIT")
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    n, m = a.genes, a.samples
    cfg = {"workload": f"C2: {n} genes x {m} samples per GPU, ~condition (p=2) Wald: fitDisp(MLE)+fitDisp(MAP)+fitBeta",
           "genes_per_gpu": n, "samples": m, "p": 2, "parallelism": f"gene-sharded x{world}",
           "l2": "inputs rotate over 4 device replicas (400 MB working set > 126 MB L2)"}

    if a.impl == "reference":
        if rank != 0:
            return
        T = host_threads()
        eng0 = RefEngine(T)
        w = build_workload(min(n, a.cpu_sample), m, 20260923 + 2, eng0)
        v, dt, ns, eng = time_reference(w, a.cpu_sample, max(1, a.steps), max(0, a.warmup), T, budget_s=150.0)
        v1, dt1, ns1, _ = time_reference(w, min(a.cpu_sample, 1500), 1, 0, 1, budget_s=20.0)
        cfg["cpu_sample_genes"] = ns
        print(json.dumps({
            "impl": "reference", "metric": "genes/sec, DESeq2 Wald hot path (fitDisp MLE + fitDisp MAP + fitBeta)",
            "value": v, "unit": "genes/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic (makeExampleDESeqDataSet law, PCG64 seed)", "config": cfg,
            "cpu_baseline": {"value": v, "unit": "genes/s", "cores": T, "kind": eng.kind,
                             "sample": f"each step = the three calls on the first {ns} genes of the C2 workload, {eng.what}, "
                                       f"{T} threads (contiguous gene chunks), median step {dt:.3f} s",
                             "single_thread": {"value": v1, "unit": "genes/s", "cores": 1,
                                               "sample": f"first {ns1} genes, one pass of {dt1:.2f} s"}},
            "e2e": {"value": v, "unit": "genes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    import torch
    import torch.distributed as dist
    import deseq2_b200
    from deseq2_b200 import device as D
    from deseq2_b200 import wrappers as W
    torch.cuda.set_device(local_rank)
    affinity_at_start = os.sched_getaffinity(0)
    cfg["host_library_threads"] = limit_library_thread_pools()
    cfg["numa"] = bind_to_gpu_numa_node(torch, local_rank)
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank),
                                timeout=datetime.timedelta(seconds=180))
    dev = torch.device("cuda", local_rank)
    L = deseq2_b200.lib()
    cfg["engine_library"] = os.path.basename(deseq2_b200.lib_path())   # experiment builds are named libb200nb_exp_*.so

    w = build_workload(n, m, 20260923 + 2 + 1000 * rank, W)
    ng = len(w["counts"])           # genes with a non-zero row sum: the ones that count for `value`
    if world > 1 and ng < n:
        # equal shard shapes for the all-gather: top the shard up to n rows by repeating its first genes
        # (extra work that is NOT counted in `value`)
        idx = np.r_[np.arange(ng), np.arange(n - ng) % ng]
        for k in ("counts", "mu", "nf", "log_alpha0", "log_dispInit", "log_dispFit", "dispersion", "beta0"):
            w[k] = np.asfortranarray(w[k][idx])
    nrow = len(w["counts"])
    p = w["x"].shape[1]
    NREP = 4
    reps = []
    xd = D.x_to_device(w["x"], dev)
    for _ in range(NREP):
        reps.append(dict(
            y=D.to_gene_major(w["counts"], dev), mu=D.to_gene_major(w["mu"], dev),
            la0=torch.as_tensor(w["log_alpha0"], device=dev), lai=torch.as_tensor(w["log_dispInit"], device=dev),
            lfit=torch.as_tensor(w["log_dispFit"], device=dev), disp=torch.as_tensor(w["dispersion"], device=dev),
            beta0=torch.as_tensor(np.ascontiguousarray(w["beta0"].T), device=dev)))
    sfd = torch.as_tensor(w["sf"], device=dev)
    contrast = torch.as_tensor(np.r_[1.0, np.zeros(p - 1)], device=dev)
    lamd = torch.as_tensor(w["lam"], device=dev)
    outs = [None, None, None]
    # per-step result exchange (N > 1): beta, beta_var, log dispersion, padded to n genes per rank
    # the kernels write beta (p x n), Var beta (p x n) and the MAP log-dispersion (n) straight into `packed`
    # Two buffer sets alternate so the all-gather of step k (asynchronous, NCCL's own stream) overlaps the kernels of
    # step k+1; a buffer is reused only after its previous gather has completed.
    NBUF = 2
    gathered = [torch.empty((world, 2 * p + 1, nrow), dtype=torch.float64, device=dev) for _ in range(NBUF)] if world > 1 else None
    packs = [torch.zeros((2 * p + 1, nrow), dtype=torch.float64, device=dev) for _ in range(NBUF)] if world > 1 else None
    pending = [None] * NBUF

    outs_b = None
    if world > 1:
        f64 = lambda *sh: torch.empty(sh, dtype=torch.float64, device=dev)
        ldd = D.ld_for(m)
        shared1 = {k: f64(nrow) for k in ("last_change", "initial_lp", "initial_dlp", "last_lp", "last_dlp", "last_d2lp")}
        shared1.update(iter=torch.empty(nrow, dtype=torch.int32, device=dev),
                       iter_accept=torch.empty(nrow, dtype=torch.int32, device=dev))
        shared2 = dict(iter=f64(nrow), contrast_num=f64(nrow), contrast_denom=f64(nrow), deviance=f64(nrow),
                       hat_diagonals=f64(nrow, ldd), mu=f64(nrow, ldd))
        outs_b = [(dict(shared1, log_alpha=pk[2 * p]), dict(shared2, beta_mat=pk[:p], beta_var_mat=pk[p:2 * p]))
                  for pk in packs]
    ev = lambda: torch.cuda.Event(enable_timing=True)
    cpu_times = []
    kern_ms = {"fit_disp_mle": 0.0, "fit_disp_map": 0.0, "fit_beta": 0.0}

    def step(i, timed, comm=True):
        r = reps[i % NREP]
        if world > 1:
            b = i % NBUF
            if pending[b] is not None:      # this buffer's previous all-gather must be done before it is rewritten
                pending[b].wait()
                pending[b] = None
            outs[1], outs[2] = outs_b[b]
        e = [ev() for _ in range(4)] if timed else None
        cpu_t = [time.perf_counter()]
        if timed:
            e[0].record()
        outs[0] = D.fit_disp(r["y"], xd, r["mu"], r["la0"], r["la0"], 1.0, MIN_LOG_ALPHA, 1.0, 1e-6, 100, False,
                             m=m, out=outs[0])
        cpu_t.append(time.perf_counter())
        if timed:
            e[1].record()
        outs[1] = D.fit_disp(r["y"], xd, r["mu"], r["lai"], r["lfit"], w["priorVar"], MIN_LOG_ALPHA, 1.0, 1e-6, 100,
                             True, m=m, out=outs[1])
        cpu_t.append(time.perf_counter())
        if timed:
            e[2].record()
        outs[2] = D.fit_beta(r["y"], xd, sfd, r["disp"], contrast, r["beta0"], lamd, 1e-8, 100, out=outs[2])
        cpu_t.append(time.perf_counter())
        cpu_times.append(cpu_t)
        if timed:
            e[3].record()
        if world > 1 and comm:
            pending[b] = dist.all_gather_into_tensor(gathered[b], packs[b], async_op=True)
        return e

    # the sampler thread is started BEFORE the warm-up so its start-up (GIL hand-over) cannot delay the first timed
    # launches; samples are attributed to the timed region by timestamp afterwards
    sampler = ClockSampler(local_rank)
    if rank == 0 and not os.environ.get("B200NB_NO_SAMPLER"):
        sampler.start()
    for i in range(max(a.warmup, 3)):
        step(i, True)            # warm-up includes the event records the timed steps make
    torch.cuda.synchronize()
    launches0 = L.b200nb_kernel_launches()
    # The K timed steps run in up to WINDOWS consecutive windows (each between barrier + synchronize) and the per-step
    # time of the MEDIAN window is reported (all windows are listed in config.timed_windows_ms): the GPU boxes show an
    # occasional ~80 ms stall that is unrelated to the workload (it hits whatever kernel happens to be running,
    # also with garbage collection off and zero cudaMalloc/cudaFree traffic), and a single timed region would
    # otherwise be at its mercy.
    WINDOWS = min(3, a.steps)
    bounds = [a.steps * k // WINDOWS for k in range(WINDOWS + 1)]
    no_ev = bool(os.environ.get("B200NB_NO_STEP_EVENTS"))
    win_ms, evs = [], []
    for k in range(WINDOWS):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t_start, t_end = ev(), ev()
        w0 = time.perf_counter()
        if k == 0:
            w0_first = w0
        t_start.record()
        evs += [step(i, not no_ev) for i in range(bounds[k], bounds[k + 1])]
        for b_ in range(NBUF if world > 1 else 0):   # the timed region ends when every gather has landed
            if pending[b_] is not None:
                pending[b_].wait()
                pending[b_] = None
        t_end.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        tm = torch.tensor([t_start.elapsed_time(t_end)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        win_ms.append(float(tm.item()))
    # the steps that keep the clock sampler busy below rewrite `outs`: keep a device copy of the last timed step's
    # results; the host copy and the sampling happen after the sampler has stopped
    last_outs = [{k: t.clone() for k, t in d.items() if t is not None} for d in outs] \
        if a.dump_outputs and rank == 0 else None
    w0 = w0_first
    w0_wall = time.time() - (time.perf_counter() - w0)
    launches = L.b200nb_kernel_launches() - launches0
    per_step = sorted(t / (bounds[k + 1] - bounds[k]) for k, t in enumerate(win_ms))
    cfg["timed_windows_ms"] = [round(v, 3) for v in win_ms]
    cfg["timed_window_reported"] = "per-step time of the median of %d windows that split the K timed steps" % WINDOWS
    # keep the GPU busy a little longer so the clock sampler sees load even for very short runs
    clocks = None
    if rank == 0:
        t_extra = time.time()
        i = 0
        while sampler.proc is not None and len(sampler.rows_since(w0_wall)) < 2 and time.time() - t_extra < 1.5:
            step(i, False, comm=False)   # rank-local only: no collectives outside the lock-step region
            i += 1
            if i % 8 == 0:
                torch.cuda.synchronize()
        torch.cuda.synchronize()
        sampler.window = (w0_wall, time.time())
        clocks = sampler.stop()
    dumped = last_step_outputs(last_outs, ng, m) if last_outs is not None else None
    if no_ev:
        evs = []
        kern_ms = {"fit_disp_mle": 1e-9, "fit_disp_map": 1e-9, "fit_beta": 1e-9}
    if os.environ.get("B200NB_BENCH_DEBUG") and rank == 0 and not no_ev:
        ct = cpu_times[max(a.warmup, 3):max(a.warmup, 3) + a.steps]
        print("cpu enqueue ms per call (max over steps):", [round(1e3 * max(c[k + 1] - c[k] for c in ct), 3) for k in range(3)],
              "cpu total enqueue ms:", round(1e3 * (ct[-1][3] - ct[0][0]), 2), "gpu ms:", round(sum(win_ms), 2), file=sys.stderr)
        print("cpu per-step [mle,map,beta] ms:", [[round(1e3 * (c[k + 1] - c[k]), 2) for k in range(3)] for c in ct], file=sys.stderr)
        print("per-step ms:", [[round(e[k].elapsed_time(e[k + 1]), 3) for k in range(3)] for e in evs], file=sys.stderr)
    for e in evs:
        kern_ms["fit_disp_mle"] += e[0].elapsed_time(e[1]) / a.steps
        kern_ms["fit_disp_map"] += e[1].elapsed_time(e[2]) / a.steps
        kern_ms["fit_beta"] += e[2].elapsed_time(e[3]) / a.steps
    if world > 1:
        ngt = torch.tensor([ng], dtype=torch.float64, device=dev)
        dist.all_reduce(ngt, op=dist.ReduceOp.SUM)
        total_genes = float(ngt.item())
    else:
        total_genes = float(ng)
    ms_per_step = per_step[WINDOWS // 2]
    value = total_genes / (ms_per_step * 1e-3)

    # ---- e2e through the C ABI with host buffers (rank-local, then max over ranks)
    e2e = None
    if not a.no_e2e:
        import ctypes
        # every step is a NEW DESeq() run: b200nb_cache_clear() first, so nothing uploaded by an earlier step can be
        # reused; within the step the library recognises (by content hash) the count matrix it is handed three times
        # and the fitted means it is handed twice, and uploads each once.  Bytes are the library's own counters.
        for _ in range(2):
            L.b200nb_cache_clear()
            three_calls_host(w, W)
        ke = max(3, min(a.steps, 10))
        if world > 1:
            dist.barrier()
        st0 = (ctypes.c_longlong * 6)()
        L.b200nb_host_stats(st0, 6)
        per = []
        for _ in range(ke):
            t0 = time.perf_counter()
            L.b200nb_cache_clear()
            res = three_calls_host(w, W)
            per.append(time.perf_counter() - t0)
            del res                         # the results are released outside the timed region (R's gc runs later too)
        allt = torch.tensor([float(np.median(per))], dtype=torch.float64, device=dev)
        if world > 1:
            gl = [torch.zeros_like(allt) for _ in range(world)]
            dist.all_gather(gl, allt)
            cfg["e2e_ms_per_rank"] = [round(float(t.item()) * 1e3, 2) for t in gl]
        st1 = (ctypes.c_longlong * 6)()
        L.b200nb_host_stats(st1, 6)
        dt = float(np.median(per))      # median step
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e = {"value": total_genes / float(tt.item()), "unit": "genes/s",
               "h2d_bytes_per_step": int((st1[0] - st0[0]) // ke), "d2h_bytes_per_step": int((st1[1] - st0[1]) // ke),
               "host_bytes_hashed_per_step": int((st1[5] - st0[5]) // ke),
               "bytes_served_from_device_cache_per_step": int((st1[4] - st0[4]) // ke),
               "caller_buffer_bytes_per_step": {"in": host_bytes(ng, m, p)[0], "out": host_bytes(ng, m, p)[1]},
               "ms_per_step": float(tt.item()) * 1e3, "steps": ke, "statistic": "median step",
               "what": "b200nb_fit_disp x2 + b200nb_fit_beta with host (R-layout, pageable) buffers through "
                       "deseq2_b200.wrappers; device cache cleared at the start of every step; within a step the count "
                       "matrix (passed 3x) and the fitted means (2x) are uploaded once (content-hash hit), the "
                       "normalisation-factor matrix is recognised as a replicated size-factor vector"}

    # ---- the whole DESeq() Wald path on the device (pre-steps, both dispersion fits, trend, grid refits, Wald fit and
    # statistics; counts resident in HBM): reported next to `value`, which stays the three hot-path calls
    full = None
    try:
        from deseq2_b200 import device_pipeline as DP
        yfull = D.to_gene_major(np.ascontiguousarray(w["counts"][:ng]), dev)
        for _ in range(2):
            DP.DESeq_device(yfull, w["x"], w["sf"])
        torch.cuda.synchronize()
        perf_ = []
        for _ in range(7):
            t0 = time.perf_counter()
            DP.DESeq_device(yfull, w["x"], w["sf"])
            torch.cuda.synchronize()
            perf_.append(time.perf_counter() - t0)
        dtf = float(np.median(perf_))
        tt = torch.tensor([dtf], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        full = {"value": total_genes / float(tt.item()), "unit": "genes/s", "ms_per_step": float(tt.item()) * 1e3,
                "what": "device_pipeline.DESeq_device: prep kernel + fitDisp MLE + grid refit + trend kernel + fitDisp MAP "
                        "+ grid refit + fitBeta + Wald statistics, counts resident in HBM, wall clock incl. host syncs"}
    except Exception as ex:  # pragma: no cover
        full = {"error": repr(ex)[:200]}
    # The same analysis the way R's DESeq() runs it by default: size factors estimated from the raw counts (on the
    # device) and count outliers replaced and refitted (minReplicatesForReplace = 7).  Those code paths have only been
    # verified under the SIMT emulator so far, so they are timed in a child process (own CUDA context, hard timeout):
    # whatever happens there cannot disturb the numbers above.
    if rank == 0 and isinstance(full, dict) and "value" in full:
        try:
            import subprocess
            env = dict(os.environ)
            for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT"):
                env.pop(k, None)
            env["CUDA_VISIBLE_DEVICES"] = os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",")[local_rank] \
                if os.environ.get("CUDA_VISIBLE_DEVICES") else str(local_rank)
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--r-default-probe", "--genes", str(n),
                                "--samples", str(m)], env=env, capture_output=True, text=True, timeout=240)
            full["r_default"] = json.loads(r.stdout.strip().splitlines()[-1]) if r.returncode == 0 else \
                {"error": (r.stderr or r.stdout)[-200:]}
        except Exception as ex:  # pragma: no cover
            full["r_default"] = {"error": repr(ex)[:200]}

    cfgs = None
    if not a.no_configs:
        try:
            pk = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs", 6650.0))
        except Exception:
            pk = 6650.0
        cfgs = configs_block(world, rank, dev, pk, quick=a.quick_configs)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    dom = max(kern_ms, key=kern_ms.get)
    if dom.startswith("fit_disp"):
        alg_bytes = ng * (12 * m + 88)
    else:
        alg_bytes = ng * (20 * m + 24 * p + 40)
    achieved = alg_bytes / (kern_ms[dom] * 1e-3) / 1e9
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(dom)
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic,
                "peak_source": "MEASURED_PEAKS.json (of measured)" if peaks else "fallback 6650 GB/s (of fallback)",
                "kernel_ms": kern_ms, "alg_bytes_per_launch": alg_bytes,
                "note": "fp64 transcendental-bound path (~300 flop/B): HBM fraction is small by construction; the "
                        "binding unit is the FP64 pipe (ncu summaries under profiles/)"}

    cpu = None
    if not a.no_cpu_baseline:
        os.sched_setaffinity(0, affinity_at_start)     # the CPU baseline gets every host thread, not one NUMA node
        cpu = cpu_baseline_record(w, a.cpu_sample, 3, 1)

    line = {"metric": "genes/sec, DESeq2 Wald hot path (fitDisp MLE + fitDisp MAP + fitBeta)", "value": value,
            "unit": "genes/s", "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic (makeExampleDESeqDataSet law, PCG64 seed 20260925)", "config": cfg,
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu,
            "full_pipeline": full, "genes_fitted": total_genes, "configs": cfgs}
    print(json.dumps(line))
    if dumped is not None:
        os.makedirs(a.dump_outputs, exist_ok=True)
        for name, v in dumped.items():
            np.save(os.path.join(a.dump_outputs, name + ".npy"), v)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
