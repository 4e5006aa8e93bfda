"""Stored outputs of the reference's own src/DESeq2.cpp, for the tests that compare with it.

oracle/_ref/libdeseq2_ref.so is that translation unit compiled unchanged against the stand-in headers of
oracle/ref_standin/ (oracle/ref.py); it can only be built where the reference source is at hand.  What it returned for
the tests' seeded inputs is kept under tests/golden/reference/, so the comparisons run on any checkout.  The CPU
comparisons keep every gene of every call; the -m gpu module keeps a seeded sample of GPU_ROWS genes per call (every
gene of a smaller call).  hat_diagonals keeps a seeded sample of COLS sample columns.  Each call also keeps a
fingerprint of its inputs, checked before its outputs are used, and each file records the sha256 of the src/DESeq2.cpp
it was recorded from (source_sha256).

To store them again (needs oracle/_ref/libdeseq2_ref.so; the -m gpu module may run on the SIMT-emulated engine):

    B200NB_RECORD_REFERENCE=1 python -m pytest tests/test_oracle_vs_reference.py
    B200NB_RECORD_REFERENCE=1 python -m pytest tests/test_emulated_kernels.py -k reference
    B200NB_RECORD_REFERENCE=1 B200NB_LIB=tests/simt_emu/_build/libb200nb_emu.so \
        python -m pytest tests/test_parity_reference_gpu.py -m gpu
"""
import inspect
import json
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference")
RECORD = os.environ.get("B200NB_RECORD_REFERENCE") == "1"
GPU_ROWS = 400                                                    # genes kept per call of the -m gpu module
ROWS = {"parity_reference_gpu": GPU_ROWS}                         # per store; every gene elsewhere
COLS = 16                                                         # hat_diagonals columns kept per call
_cache = {}


def _fingerprint(kw):
    fp = []
    for k in sorted(kw):
        v = kw[k]
        if v is None:
            fp.append(np.nan)
        else:
            a = np.asarray(v, dtype=np.float64)
            fp += [a.size, float(np.sum(a))]
    return np.array(fp)


def _load(path):
    """{"<case>#<call>/<output>": array}.  On disk: one flat float64 vector, byte-shuffled (all first bytes, then all
    second bytes, ...) so that it compresses, a JSON index of offsets and shapes, and source_sha256."""
    if path not in _cache:
        store = {}
        if os.path.exists(path):
            z = np.load(path)
            data = np.ascontiguousarray(z["data"].reshape(8, -1).T).view(np.float64).ravel()
            for k, (o, shape, dt) in json.loads(str(z["index"])).items():
                store[k] = data[o:o + int(np.prod(shape))].reshape(shape).astype(dt)
        _cache[path] = store
    return _cache[path]


def _source_sha256():
    """Hash of the src/DESeq2.cpp that oracle/_ref/libdeseq2_ref.so was compiled from (written by oracle/Makefile)."""
    from oracle import ref as R
    with open(os.path.join(os.path.dirname(R._SO), "SOURCE.sha256")) as f:
        return f.read().split()[0]


def _save(path, store):
    index, parts, o = {}, [], 0
    for k in sorted(store):
        v = np.asarray(store[k])
        index[k] = (o, list(v.shape), "int32" if v.dtype.kind in "iu" else "float64")
        parts.append(v.astype(np.float64).ravel())
        o += v.size
    data = np.concatenate(parts).view(np.uint8).reshape(-1, 8).T.ravel()
    os.makedirs(os.path.dirname(path), exist_ok=True)
    np.savez_compressed(path, data=data, index=np.array(json.dumps(index)), source_sha256=np.array(_source_sha256()))


class Reference:
    """Stands in for oracle.ref in one test case: returns the stored outputs of the case's calls in call order,
    restricted to the stored genes (`rows`) and hat_diagonals columns (`cols`).  With B200NB_RECORD_REFERENCE=1 it
    calls the reference library instead and stores what it returns."""

    def __init__(self, store, case):
        self.path = os.path.join(GOLDEN, store + ".npz")
        self.rows = ROWS.get(store)
        self.case, self.calls = case, 0

    def fitDisp(self, *args, **kw):
        return self._call("fitDisp", args, kw)

    def fitDispGrid(self, *args, **kw):
        return self._call("fitDispGrid", args, kw)

    def fitBeta(self, *args, **kw):
        return self._call("fitBeta", args, kw)

    def _call(self, fn, args, kw):
        from oracle import ref as R
        kw = dict(inspect.signature(getattr(R, fn)).bind(*args, **kw).arguments)
        kw.pop("nthreads", None)            # outputs are recorded from one unchunked call of the reference
        key = f"{self.case}#{self.calls}"
        self.calls += 1
        fp = _fingerprint(kw)
        store = _load(self.path)
        if RECORD:
            out = getattr(R, fn)(**kw)
            n = len(kw["ySEXP"])
            rng = np.random.default_rng(n)
            k = None if fn == "fitDispGrid" else self.rows
            rows = np.arange(n) if k is None or n <= k else np.sort(rng.choice(n, k, replace=False))
            rec = {"fingerprint": fp, "rows": rows}
            for k, v in out.items():
                rec[k] = np.asarray(v)[rows]
            if "hat_diagonals" in rec and rec["hat_diagonals"].shape[1] > COLS:
                rec["cols"] = np.sort(rng.choice(rec["hat_diagonals"].shape[1], COLS, replace=False))
                rec["hat_diagonals"] = rec["hat_diagonals"][:, rec["cols"]]
            for k in [k for k in store if k.startswith(key + "/")]:
                del store[k]
            store.update((f"{key}/{k}", v) for k, v in rec.items())
            _save(self.path, store)
        rec = {k[len(key) + 1:]: v for k, v in store.items() if k.startswith(key + "/")}
        assert rec, f"{os.path.basename(self.path)} holds no reference output for {key}"
        assert np.allclose(rec.pop("fingerprint"), fp, rtol=1e-9, atol=0, equal_nan=True), \
            f"{key}: the inputs are not those the stored reference output was computed from"
        return rec


def take(d, r):
    """The genes (and hat_diagonals columns) of the full output `d` that the stored reference output `r` keeps."""
    out = {}
    for k, v in d.items():
        v = np.asarray(v)
        if v.ndim:
            v = v[r["rows"]]
            if k == "hat_diagonals" and "cols" in r:
                v = v[:, r["cols"]]
        out[k] = v
    return out
