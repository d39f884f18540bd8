"""Stored outputs of the original project (the compiled reference rasterizer under oracle/_ref, its simple-knn, its
Python code) for the tests that compare against it, kept in tests/golden/reference_outputs.npz.

Full-size outputs do not fit in the repository, so each one is kept as a fingerprint:
  * ``equal`` comparisons: a SHA-256 digest of the array's dtype, shape and bytes (bit-exact, as torch.equal on the
    raw bits);
  * tolerance comparisons: the values at a fixed seeded sample of at most SAMPLE flat positions (all of them for
    smaller arrays), and of the whole array its max |value| (the scale the tolerances are relative to), its sum and
    the sum of its |values|.  The sums pin the entries outside the sample: the tolerances bound the per-entry
    differences, so they also bound the difference of the sums.

Regenerating: with SGB_RECORD_REFERENCE=<file.npz> set, a test runs the original live (the GPU tests on a machine where
oracle/build.py has compiled oracle/_ref/; the CPU tests read the original's source tree, named by
SGB_REFERENCE_TREE) and ``put``s its outputs.  The comparisons then check against these fresh fingerprints, and at exit
the stored file, with the recorded cases replaced by what their comparisons read, is written to <file.npz>."""
from __future__ import annotations

import atexit
import hashlib
import os

import numpy as np
import torch

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_outputs.npz")
RECORD = os.environ.get("SGB_RECORD_REFERENCE")
SAMPLE = 1024

_stored = None
_recorded = {}      # recording runs: every fingerprint part of the live outputs
_used = set()       # ... and the keys the comparisons read


def _data():
    global _stored
    if _stored is None:
        _stored = dict(np.load(PATH)) if os.path.exists(PATH) else {}
    return _stored


def _case_of(key):
    return key.split("/", 1)[0]


def _write():
    cases = {_case_of(k) for k in _recorded}
    out = {k: v for k, v in _data().items() if _case_of(k) not in cases}
    out.update({k: _recorded[k] for k in _used})
    np.savez_compressed(RECORD, **out)


if RECORD:
    atexit.register(_write)


def _np(x):
    if isinstance(x, torch.Tensor):
        return x.detach().contiguous().cpu().numpy()
    return np.ascontiguousarray(np.asarray(x))


def digest(x) -> str:
    a = _np(x)
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return h.hexdigest()


def sample_index(n: int) -> np.ndarray:
    """The flat positions kept of an n-element array: fixed by n alone."""
    if n <= SAMPLE:
        return np.arange(n)
    return np.unique(np.random.default_rng(n).integers(0, n, SAMPLE))


def _sums(t: torch.Tensor):
    """(sum, sum of |values|) of the whole array in float64."""
    return float(torch.sum(t, dtype=torch.float64)), float(torch.sum(t.abs(), dtype=torch.float64))


class Reference:
    """The original's outputs for one test case (`case` names the inputs, e.g. the test and its parameters)."""

    def __init__(self, case: str):
        self.case = case
        self.recording = bool(RECORD)

    def _key(self, name, kind):
        return f"{self.case}/{name}/{kind}"

    def _get(self, name, kind):
        k = self._key(name, kind)
        src = _recorded if self.recording else _data()
        if k not in src:
            raise KeyError(f"no stored reference output {k} in {PATH}")
        _used.add(k)
        return src[k]

    def put(self, name: str, x) -> None:
        """Record one output of the original (recording runs only)."""
        assert self.recording, "put() needs SGB_RECORD_REFERENCE"
        a = _np(x)
        _recorded[self._key(name, "digest")] = np.array(digest(a))
        _recorded[self._key(name, "shape")] = np.array(a.shape, np.int64)
        if a.dtype.kind == "f":
            flat = torch.from_numpy(a.reshape(-1))
            _recorded[self._key(name, "sample")] = a.reshape(-1)[sample_index(flat.numel())]
            _recorded[self._key(name, "absmax")] = np.float64(flat.abs().max()) if flat.numel() else np.float64(0)
            _recorded[self._key(name, "sums")] = np.array(_sums(flat), np.float64)

    def equal(self, name: str, got) -> bool:
        """Bit-exact equality with the original's output."""
        return digest(got) == str(self._get(name, "digest"))

    def pair(self, name: str, got):
        """(ours, the original's) at the stored sample positions, float64, and the original's max |value|."""
        shape = tuple(int(s) for s in self._get(name, "shape"))
        assert tuple(got.shape) == shape, (self.case, name, tuple(got.shape), shape)
        got = got if isinstance(got, torch.Tensor) else torch.from_numpy(_np(got))
        flat = got.detach().reshape(-1)
        a = flat[torch.as_tensor(sample_index(flat.numel()), device=flat.device)].double().cpu()
        b = torch.from_numpy(self._get(name, "sample").astype(np.float64))
        return a, b, float(self._get(name, "absmax"))

    def _sum_gap(self, name, got):
        """(|sum(ours) - sum(original)|, sum |original|, number of entries)."""
        s, abs_s = (float(v) for v in self._get(name, "sums"))
        got = got if isinstance(got, torch.Tensor) else torch.from_numpy(_np(got))
        return abs(_sums(got.detach().reshape(-1))[0] - s), abs_s, got.numel()

    def frac_bad(self, name: str, got, rtol=1e-4, atol_scale=1e-4) -> float:
        """util.frac_bad (share of entries with |a-b| > rtol*|b| + atol_scale*max|b|) on the sample; at least one
        entry of the whole array (1/n) when the sums differ by more than those per-entry bounds add up to."""
        a, b, m = self.pair(name, got)
        frac = float(((a - b).abs() > rtol * b.abs() + atol_scale * m).double().mean())
        gap, abs_s, n = self._sum_gap(name, got)
        if gap > (rtol * abs_s + atol_scale * m * n) * (1 + 1e-9):
            frac = max(frac, 1.0 / n)
        return frac

    def rel_err(self, name: str, got) -> float:
        """util.rel_err (max |a-b| / max|b|) on the sample, or the mean difference the sums imply if that is larger."""
        a, b, m = self.pair(name, got)
        gap, _, n = self._sum_gap(name, got)
        return max(float((a - b).abs().max()), gap / n) / (m + 1e-30)
