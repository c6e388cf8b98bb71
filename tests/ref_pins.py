"""What the verbatim reference build (oracle/_ref) returned for the inputs of the pinning tests, stored in
tests/golden/ref_pins.json so that those comparisons run everywhere, without the reference sources.

A test asks `pinned(key, compute)` for the reference's result and compares its own (restated or product) result with it
through `digest`. Arrays of up to 64 elements are stored as values, longer ones as dtype-normalised SHA-256 digests.
Re-record after a change of test inputs, with oracle/_ref built (make -C oracle ref):
    JAERO_RECORD_REF_PINS=1 python -m pytest tests/test_fec_pinning.py tests/test_oracle_golden.py tests/test_reassembly.py"""
import hashlib
import json
import os

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_pins.json")
RECORD = os.environ.get("JAERO_RECORD_REF_PINS") == "1"
_pins = None


def digest(x):
    """JSON-able form of a result: small arrays as lists, large ones as 'shape:sha256' of the int64 / float64 bytes"""
    if isinstance(x, np.ndarray):
        a = np.ascontiguousarray(x, dtype="<f8" if x.dtype.kind == "f" else "<i8")
        if a.size <= 64:
            return a.tolist()
        return "%s:%s" % ("x".join(map(str, a.shape)), hashlib.sha256(a.tobytes()).hexdigest())
    if isinstance(x, (list, tuple)):
        return [digest(v) for v in x]
    if isinstance(x, dict):
        return {str(k): digest(v) for k, v in x.items()}
    if isinstance(x, (bytes, bytearray)):
        return bytes(x).hex()
    if isinstance(x, (bool, np.bool_)):
        return bool(x)
    if isinstance(x, np.integer):
        return int(x)
    if isinstance(x, np.floating):
        return float(x)
    return x


def pinned(key, compute):
    """The reference's result for `key` in digest form: from the golden file, or computed by `compute()` and stored there
    when recording."""
    global _pins
    if _pins is None:
        _pins = {}
        if os.path.exists(PATH):
            with open(PATH) as fh:
                _pins = json.load(fh)
    if RECORD:
        _pins[key] = json.loads(json.dumps(digest(compute())))
        with open(PATH, "w") as fh:
            json.dump(_pins, fh, indent=0, sort_keys=True)
    assert key in _pins, "no reference result stored for %s (record with JAERO_RECORD_REF_PINS=1)" % key
    return _pins[key]


def same(got, key, compute):
    """got (digested) equals the reference's stored result for key"""
    return json.loads(json.dumps(digest(got))) == pinned(key, compute)
