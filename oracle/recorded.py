"""Outputs of the pinned reference build (oracle/_ref), recorded on a B200, so that the parity tests run where neither
the reference's sources nor its build exist.

TEST INFRASTRUCTURE.  tests/golden/reference_outputs.json maps "<test file>::<test name[parameters]>" to what the
reference computed for that test: for each output array its shape, the SHA-256 of its float32 bit patterns (every NaN
folded to one pattern, so that equal digests mean what conftest.bits_equal == 0 means) and a fixed sample of its elements
(for a count of differing elements when the digests differ); plain numbers, such as the reference's printed run time, as
they are.  "_recorded_on" names the GPU and power limit those times were measured at.

To record again (needs a GPU and oracle/_ref built by oracle/build_ref.sh), run the GPU tests with
GIPUMA_RECORD_REFERENCE set to a JSON file: each test then runs the live reference, adds its entry to that file and
compares against it as usual.  Copy the file to tests/golden/reference_outputs.json afterwards.
"""
from __future__ import annotations

import base64
import hashlib
import json
import os
import subprocess

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden",
                      "reference_outputs.json")
SAMPLE = 128
_golden = None


def _bits(a) -> np.ndarray:
    a = np.ascontiguousarray(a, dtype=np.float32)
    u = a.view(np.uint32).ravel().copy()
    u[np.isnan(a).ravel()] = 0x7FC00000
    return u


def _sample_index(n: int) -> np.ndarray:
    return np.sort(np.random.default_rng(n).choice(n, min(n, SAMPLE), replace=False))


def digest(a) -> dict:
    u = _bits(a)
    return {"shape": list(np.shape(a)), "sha256": hashlib.sha256(u.tobytes()).hexdigest(),
            "sample": base64.b64encode(u[_sample_index(u.size)].astype("<u4").tobytes()).decode()}


def _device() -> dict:
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().split(", ")
    return {"gpu": q[0], "power_limit": q[1] if len(q) > 1 else None}


class Recorded:
    """The reference's outputs for one test."""

    def __init__(self, key: str, entry: dict):
        self.key, self.entry = key, entry

    def __getitem__(self, name: str) -> float:
        return self.entry[name]

    def _compare(self, name, ours):
        rec = self.entry[name]
        assert list(np.shape(ours)) == rec["shape"], "%s %s: shape %s, the reference's %s" % (
            self.key, name, list(np.shape(ours)), rec["shape"])
        u = _bits(ours)
        sample = np.frombuffer(base64.b64decode(rec["sample"]), dtype="<u4")
        return u, rec, int((u[_sample_index(u.size)] != sample).sum()), sample.size

    def bits_differ(self, name: str, ours) -> int:
        """0 iff `ours` has the bit patterns of the reference's output `name` (NaN == NaN); otherwise the number of
        differing elements in the recorded sample, at least 1."""
        u, rec, n, _ = self._compare(name, ours)
        return 0 if hashlib.sha256(u.tobytes()).hexdigest() == rec["sha256"] else max(1, n)

    def fraction_differing(self, name: str, ours) -> float:
        """Fraction of the recorded sample of output `name` whose bit patterns differ from `ours`."""
        _, _, n, m = self._compare(name, ours)
        return n / m


def reference(node, run) -> Recorded:
    """The reference's outputs for the pytest item `node`.  `run()` computes them on the live reference build and
    returns {name: array or number}; it is called only when recording (GIPUMA_RECORD_REFERENCE)."""
    global _golden
    key = "%s::%s" % (node.path.name, node.name)
    out = os.environ.get("GIPUMA_RECORD_REFERENCE")
    if out:
        data = json.load(open(out)) if os.path.exists(out) else {"_recorded_on": _device()}
        data[key] = {k: digest(v) if isinstance(v, np.ndarray) else float(v) for k, v in run().items()}
        with open(out, "w") as fh:
            json.dump(data, fh, indent=1, sort_keys=True)
            fh.write("\n")
    else:
        if _golden is None:
            with open(GOLDEN) as fh:
                _golden = json.load(fh)
        data = _golden
    assert key in data, "no recorded reference output for %s in %s" % (key, out or GOLDEN)
    return Recorded(key, data[key])
