"""What tests/test_ref_ops_gpu.py and tests/test_integration_gpu.py compare with when the original project's compiled
ops (oracle/_ref, built by oracle/build_ref.py from the original sources, which are not part of this repository) are
absent: pins of the original ops' outputs on the tests' seeded inputs, stored in tests/golden/ref_ops.npz.

A bit-exact output is pinned by the SHA-256 of its dtype, shape and bytes, next to its shape and a fixed, seeded sample
of 1024 of its values (which say where a failing output differs); any other output by its shape, its largest
magnitude and such a sample, checked with the test's tolerance.

    VSR_RECORD_REF_PINS=<file.npz> python -m pytest tests/test_ref_ops_gpu.py tests/test_integration_gpu.py

records the pins from the compiled original ops while the tests compare with them as usual (a GPU and oracle/_ref with
its pyref/ wrappers are needed; recording fails without them).

Provenance of the committed file: the original sources were not at hand when it was made, so its pins were taken from
this project's C oracle and kernels at the code of profiles/gpu_tests_r02j.log.  That run collected 188 GPU tests,
these among them, and all 188 passed against the compiled original ops; the oracle, the kernels and these tests'
inputs have not changed since.  On these inputs the pinned outputs therefore equal the original's bit for bit where a
test compares bit for bit, and lie within the test's tolerance of it elsewhere.  Those pins carry no value sample next
to their hash.  Re-record the file wherever the original ops can be built.
"""
import atexit
import hashlib
import os

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_ops.npz")
RECORD = os.environ.get("VSR_RECORD_REF_PINS")
SAMPLES = 1024
_recorded = {}
_pins = None


def _np(a):
    return a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)


def _pin(key, default=None):
    global _pins
    if _pins is None:
        with np.load(PATH) as z:
            _pins = {k: z[k] for k in z.files}
    if default is None:
        assert key in _pins, f"no pin {key} in {PATH}"
    return _pins.get(key, default)


def _digest(a):
    a = np.ascontiguousarray(a)
    return hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).hexdigest()


def _sample(case, n):
    seed = int(hashlib.sha256(case.encode()).hexdigest()[:8], 16)
    return np.sort(np.random.default_rng(seed).choice(n, size=min(n, SAMPLES), replace=False))


def _record(case, want, exact):
    assert RECORD, case
    pins = {case + "/shape": np.array(want.shape), case + "/values": want.reshape(-1)[_sample(case, want.size)]}
    if exact:
        pins[case + "/sha256"] = np.array(_digest(want))
    else:
        pins[case + "/absmax"] = np.array(np.abs(want).max())
    for k, v in pins.items():        # every comparison recorded under one case must see the same output
        assert k not in _recorded or np.array_equal(_recorded[k], v), k
    _recorded.update(pins)


def _require_reference(case, want):
    if RECORD and want is None:
        raise AssertionError(f"{case}: recording the pins needs the original ops' output (oracle/_ref)")


def assert_equal(case, got, want=None):
    """`got` equals the original op's output for `case` bit for bit; `want` is that output when the compiled op ran."""
    got = _np(got)
    _require_reference(case, want)
    if want is not None:
        want = _np(want)
        assert np.array_equal(got, want), case
        if RECORD:
            _record(case, want, exact=True)
        return
    if _digest(got) == str(_pin(case + "/sha256")):
        return
    where = f"{got.dtype} {got.shape}"
    values = _pin(case + "/values", False)
    if values is not False and tuple(got.shape) == tuple(_pin(case + "/shape")):
        diff = np.abs(got.reshape(-1)[_sample(case, got.size)].astype(np.float64) - values)
        where += f", {int((diff != 0).sum())} of {diff.size} sampled values differ, by up to {diff.max():.3g}"
    raise AssertionError(f"{case}: differs from the original op's output ({where})")


def assert_close(case, got, want=None, rel=1e-5):
    """|got - the original op's output for `case`| <= rel * max(1, its largest magnitude), everywhere when the compiled
    op ran (`want`), else on the pinned sample; returns that tolerance."""
    got = _np(got)
    _require_reference(case, want)
    if want is not None:
        want = _np(want)
        tol = rel * max(1.0, float(np.abs(want).max()))
        assert got.shape == want.shape and np.abs(got - want).max() <= tol, case
        if RECORD:
            _record(case, want, exact=False)
        return tol
    tol = rel * max(1.0, float(_pin(case + "/absmax")))
    assert tuple(got.shape) == tuple(_pin(case + "/shape")), case
    assert np.abs(got.reshape(-1)[_sample(case, got.size)] - _pin(case + "/values")).max() <= tol, case
    return tol


@atexit.register
def _write():
    if RECORD and _recorded:
        np.savez_compressed(RECORD, **_recorded)
