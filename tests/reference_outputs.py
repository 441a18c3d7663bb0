"""Outputs of the reference's own code (oracle/_ref: its CUDA kernels, its CUDA model path and its CPU
orchestration, compiled from a reference checkout) kept as golden data, so that the bit-exactness
tests hold on a machine without a reference build.

check(ours, live, key, what) compares `ours` bit for bit with
  * `live`, the reference's output computed in the same run, when oracle/_ref is built (else None);
  * the output recorded under `key` in tests/golden/reference_outputs.json: the SHA-256 of its 32-bit
    pattern (float32; token ids as float32, exact below 2^24) and 16 sampled values that name a
    difference in the failure message.

Recording: with oracle/_ref built and KLLM_RECORD_REFERENCE=<file.json> set, the live outputs are
written to that file (starting from the stored records, replacing the keys the run reaches) instead of
being compared with the stored ones.  Copy the file to tests/golden/reference_outputs.json.
"""
import atexit
import hashlib
import json
import os

import numpy as np

from conftest import GOLDEN
from gpu_util import assert_bit_equal, bits

GOLDEN_FILE = GOLDEN / "reference_outputs.json"
RECORD_TO = os.environ.get("KLLM_RECORD_REFERENCE")
SAMPLES = 16
_stored = None
_recorded = {}


def live_reference(flavour="llama2"):
    """RefCuda for `flavour` when oracle/_ref is built, else None (recording requires the build)."""
    from oracle.binding import REF_QWEN_SO, REF_SO, RefCuda
    so = REF_SO if flavour == "llama2" else REF_QWEN_SO
    if not so.exists():
        if RECORD_TO:
            raise FileNotFoundError(f"recording reference outputs needs {so}")
        return None
    return RefCuda(flavour)


def _words(a):
    if isinstance(a, (list, tuple)):
        a = np.stack([bits(x).view(np.float32) for x in a]) if a and np.ndim(a[0]) else np.asarray(a, np.float32)
    return bits(a).ravel()


def digest(a):
    w = _words(a)
    idx = np.sort(np.random.default_rng(w.size).choice(w.size, min(SAMPLES, w.size), replace=False))
    return {"n": int(w.size), "sha256": hashlib.sha256(w.tobytes()).hexdigest(),
            "sample": [[int(i), int(w[i])] for i in idx]}


def _load():
    global _stored
    if _stored is None:
        _stored = json.loads(GOLDEN_FILE.read_text()) if GOLDEN_FILE.exists() else {}
    return _stored


def _write():
    out = dict(_load())
    out.update(_recorded)
    with open(RECORD_TO, "w") as f:  # one record per line
        f.write("{\n" + ",\n".join(f"{json.dumps(k)}: {json.dumps(out[k])}" for k in sorted(out)) + "\n}\n")


if RECORD_TO:
    atexit.register(_write)


def check(ours, live, key, what=""):
    if live is not None:
        assert_bit_equal(_words(ours).view(np.float32), _words(live).view(np.float32), f"{what} (live reference)")
    if RECORD_TO:
        if live is None:
            raise AssertionError(f"{key}: recording needs the live reference output")
        _recorded[key] = digest(live)
        return
    want = _load().get(key)
    assert want is not None, f"{what}: no reference output recorded under {key!r} in {GOLDEN_FILE.name}"
    w = _words(ours)
    if w.size == want["n"] and hashlib.sha256(w.tobytes()).hexdigest() == want["sha256"]:
        return
    bad = [(i, int(w[i]), b) for i, b in want["sample"] if i < w.size and int(w[i]) != b]
    f32 = lambda u: float(np.uint32(u).view(np.float32))  # noqa: E731
    detail = "; ".join(f"[{i}] {f32(a)!r} vs {f32(b)!r}" for i, a, b in bad[:4]) or "sampled values agree"
    raise AssertionError(f"{what}: differs from the recorded reference output {key!r} "
                         f"({w.size} vs {want['n']} values; {len(bad)}/{len(want['sample'])} samples differ: {detail})")
