"""What the reference computed on the tests' inputs, stored under tests/golden/reference/.

The tests that compare against the reference's own sources compiled in place (oracle/_ref, see oracle/Makefile) call
the `reference` fixture instead of oracle.ref_*: same functions, same arguments, but the outputs come from
tests/golden/reference/<test module>.npz, so the comparison runs wherever the reference sources are absent.  Each
test's calls are replayed in order; a SHA-256 over all of the test's inputs, stored with them, must match, so a change
of the synthetic inputs fails the test instead of comparing against outputs for other inputs.

Bulky outputs that the tests only compare for equality are stored as SHA-256 digests (image pyramids, reference
patch caches), and the per-pixel residual magnitudes of computeResiduals as an evenly spaced sample of patches.

Re-recording needs oracle/_ref (built by `build()` where the reference sources exist) and, for the GPU test modules,
a CUDA device:

    SVO_RECORD_REFERENCE=tests/golden/reference python -m pytest tests

runs the listed tests against the compiled reference and rewrites their entries in DIR/<test module>.npz.
"""
from __future__ import annotations

import dataclasses
import functools
import hashlib
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference")
RESIDUAL_SAMPLE_PATCHES = 16


def sha256(a) -> str:
    a = np.ascontiguousarray(a)
    return hashlib.sha256(a.dtype.str.encode() + str(a.shape).encode() + a.tobytes()).hexdigest()


def _feed(h, x):
    """Canonical bytes of a call argument into the hash h."""
    if isinstance(x, np.ndarray):
        h.update(f"a{x.dtype.str}{x.shape}".encode())
        h.update(np.ascontiguousarray(x).tobytes())
    elif isinstance(x, (list, tuple)):
        h.update(f"l{len(x)}".encode())
        for v in x:
            _feed(h, v)
    elif isinstance(x, dict):
        h.update(f"d{len(x)}".encode())
        for k in sorted(x):
            h.update(str(k).encode())
            _feed(h, x[k])
    elif dataclasses.is_dataclass(x):
        _feed(h, dataclasses.asdict(x))
    elif isinstance(x, (bool, np.bool_)):
        h.update(b"b1" if x else b"b0")
    elif isinstance(x, (int, np.integer)):
        h.update(f"i{int(x)}".encode())
    elif isinstance(x, (float, np.floating)):
        h.update(f"f{float(x)!r}".encode())
    elif x is None or isinstance(x, str):
        h.update(f"s{x}".encode())
    else:
        raise TypeError(f"cannot hash a {type(x).__name__} argument")


def _visible_rows(r):
    return r["ref_patch"][np.asarray(r["visible"]).astype(bool)]


def _shrink_sia(r):
    r = dict(r)
    r["visible_ref_patch_sha256"] = sha256(_visible_rows(r))
    del r["ref_patch"]
    return r


def _shrink_residuals(r):
    r = _shrink_sia(r)
    n = len(r["abs_res"])
    rows = np.unique(np.linspace(0, n - 1, min(n, RESIDUAL_SAMPLE_PATCHES)).round().astype(np.int64))
    r["abs_res_rows"], r["abs_res"] = rows, r["abs_res"][rows]
    return r


# what is stored of an output (everything the tests read, nothing more)
SHRINK = {
    "ref_image_pyramid": lambda pyr: np.array([sha256(level) for level in pyr]),
    "ref_sparse_img_align": _shrink_sia,
    "ref_sparse_residuals": _shrink_residuals,
}


def _flatten(out):
    """output -> {path: ndarray}; path "" = a bare value, "#i" = tuple element i, otherwise a dict key."""
    if isinstance(out, dict):
        return {k: np.asarray(v) for k, v in out.items()}
    if isinstance(out, tuple):
        return {f"#{i}": np.asarray(v) for i, v in enumerate(out)}
    return {"": np.asarray(out)}


def _unflatten(leaves):
    val = {k: (v.item() if v.ndim == 0 else v) for k, v in leaves.items()}
    if list(val) == [""]:
        return val[""]
    if all(k.startswith("#") for k in val):
        return tuple(val[f"#{i}"] for i in range(len(val)))
    return val


class Reference:
    """Stands in for oracle.ref_* inside one test: replays the stored outputs, or records them when `record_dir` is
    set (then every call goes to the compiled reference and the test sees exactly what is stored)."""

    def __init__(self, module: str, test: str, record_dir: str | None = None):
        self.module, self.test, self.record_dir = module, test, record_dir
        self._hash = hashlib.sha256()
        self._n_calls = 0
        self._calls = {}  # fn -> [{path: ndarray}] in call order
        if record_dir is None:
            self._stored = _load(os.path.join(GOLDEN, module + ".npz"), test)
            if self._stored is None:
                raise LookupError(f"no stored reference outputs for {module}::{test} under {GOLDEN} "
                                  "(see tests/reference_outputs.py for how to record them)")
            self._next = {fn: 0 for fn in self._stored["calls"]}

    def __getattr__(self, fn: str):
        if not fn.startswith("ref_"):
            raise AttributeError(fn)

        def call(*args, **kwargs):
            _feed(self._hash, fn)
            _feed(self._hash, list(args))
            _feed(self._hash, kwargs)
            self._n_calls += 1
            if self.record_dir is not None:
                from oracle import binding

                if binding.ref_lib() is None:
                    raise RuntimeError("recording reference outputs needs oracle/_ref (built where the reference sources exist)")
                out = getattr(binding, fn)(*args, **kwargs)
                leaves = _flatten(SHRINK.get(fn, lambda o: o)(out))
                self._calls.setdefault(fn, []).append(leaves)
                return _unflatten(leaves)
            seq = self._stored["calls"].get(fn, [])
            i = self._next.get(fn, 0)
            if i >= len(seq):
                raise LookupError(f"{self.module}::{self.test} makes more {fn} calls than were recorded ({len(seq)})")
            self._next[fn] = i + 1
            return _unflatten({k: v.copy() for k, v in seq[i].items()})

        return call

    def finish(self, records: dict):
        """End of the test: check the inputs (replay) or hand this test's record over for writing (record)."""
        digest = self._hash.hexdigest()
        if self.record_dir is not None:
            records.setdefault(self.module, {})[self.test] = dict(inputs_sha256=digest, n_calls=self._n_calls, calls=self._calls)
            return
        if self._n_calls == self._stored["n_calls"] and digest != self._stored["inputs_sha256"]:
            raise AssertionError(f"{self.module}::{self.test}: the inputs differ from those the stored reference outputs "
                                 "were recorded for")


# ---- storage: one .npz per test module; per function and output field, the values of all calls of all its tests ----
# ---- concatenated (`data`) with each call's shape (`shapes`) and test (`test`) ----
@functools.lru_cache(maxsize=None)
def _read(path):
    """{test: dict(inputs_sha256, n_calls, calls={fn: [{path: ndarray}] in call order})} of one module file."""
    if not os.path.exists(path):
        return {}
    with np.load(path, allow_pickle=False) as z:
        tests = z["tests"].tolist()
        recs = {t: dict(inputs_sha256=str(h), n_calls=int(n), calls={})
                for t, h, n in zip(tests, z["inputs_sha256"], z["n_calls"])}
        for fn in z["functions"].tolist():
            owner = z[f"{fn}|test"]
            seq = [{} for _ in owner]
            for p in z[f"{fn}|paths"].tolist():
                data, shapes, off = z[f"{fn}|{p}|data"], z[f"{fn}|{p}|shapes"], 0
                for i, shape in enumerate(shapes):
                    size = int(np.prod(shape, dtype=np.int64))
                    seq[i][p] = data[off:off + size].reshape(tuple(int(s) for s in shape))
                    off += size
            for i, t in enumerate(owner):
                recs[tests[t]]["calls"].setdefault(fn, []).append(seq[i])
    return recs


def _load(path, test):
    return _read(path).get(test)


def write(record_dir: str, records: dict):
    """Merge the recorded tests into record_dir/<module>.npz (entries of tests not recorded now are kept)."""
    os.makedirs(record_dir, exist_ok=True)
    for module, new in records.items():
        out = os.path.join(record_dir, module + ".npz")
        recs = {**_read(os.path.join(GOLDEN, module + ".npz")), **_read(out), **new}
        tests = sorted(recs)
        arrays = dict(tests=np.array(tests, dtype=str),
                      inputs_sha256=np.array([recs[t]["inputs_sha256"] for t in tests], dtype=str),
                      n_calls=np.array([recs[t]["n_calls"] for t in tests], np.int64))
        functions = sorted({fn for t in tests for fn in recs[t]["calls"]})
        arrays["functions"] = np.array(functions, dtype=str)
        for fn in functions:
            owner, seq = [], []
            for i, t in enumerate(tests):
                calls = recs[t]["calls"].get(fn, [])
                owner += [i] * len(calls)
                seq += calls
            paths = list(seq[0])
            arrays[f"{fn}|test"] = np.array(owner, np.int32)
            arrays[f"{fn}|paths"] = np.array(paths, dtype=str)
            for p in paths:
                leaves = [c[p] for c in seq]
                arrays[f"{fn}|{p}|shapes"] = np.array([l.shape for l in leaves], np.int64).reshape(len(seq), leaves[0].ndim)
                arrays[f"{fn}|{p}|data"] = np.concatenate([l.ravel() for l in leaves])
        np.savez_compressed(out, **arrays)
