import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def _ensure_oracle():
    """Build the CPU oracle library if it is missing (checker only, never the product). The reference build (oracle/_ref) is
    not needed: its results are stored under tests/golden (tests/ref_pins.py)."""
    orc = os.path.join(ROOT, "oracle", "_build", "libjaero_oracle.so")
    if not os.path.exists(orc):
        subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), "oracle"], check=True, capture_output=True)


@pytest.fixture(scope="session", autouse=True)
def oracle_libs():
    _ensure_oracle()


@pytest.fixture(scope="session")
def golden():
    import json
    with open(os.path.join(ROOT, "tests", "golden", "expected_outputs.json")) as fh:
        return json.load(fh)


def load_excerpt(name):
    import numpy as np
    return np.load(os.path.join(ROOT, "tests", "golden", name + "_excerpt.npz"))["pcm"]


def has_cuda():
    try:
        import jaero_b200
        return jaero_b200.lib().jaero_device_count() > 0
    except Exception:
        return False


def synthetic_r_packet_stream(fb, payload17, invert=False, soft_hi=230, soft_lo=25):
    """Soft-bit stream carrying one R-channel packet (19 bytes = 17 + CRC-16) the way the reference expects it
    (aerol.h:631-690 / :786-840): start-of-burst marker, filler, unique word (on both arms for OQPSK), then the 64 x 5
    interleaved block of the rate-1/2 K=7 code over the scrambled bits. Known-answer vector for the R/T layer."""
    import numpy as np
    from jaero_b200 import synth
    body = np.asarray(payload17, dtype=np.uint8)
    assert len(body) == 17
    c = synth.crc16(body)
    info = np.unpackbits(np.concatenate([body, np.array([c & 0xFF, c >> 8], dtype=np.uint8)]), bitorder="little")   # 152 bits, LSB first
    u = np.zeros(160, dtype=np.uint8)
    u[:152] = info ^ synth.scrambler_sequence(152)          # the receiver descrambles after decoding
    coded, _ = synth.conv_encode_stream(u, 0)               # tail of 8 zero input bits flushes the encoder
    block = synth.interleave(coded, 5)
    uw = np.array([(synth.UW >> (31 - i)) & 1 for i in range(32)], dtype=np.uint8)
    if int(fb) == 10500:
        uw = np.repeat(uw, 2)                               # the same word on the I and the Q arm (aerol.cpp:959-963)
    filler = np.tile(np.array([0, 0, 1, 1], dtype=np.uint8), 20)
    bits = np.concatenate([filler, uw, block, np.tile(np.array([0, 1, 1, 0], dtype=np.uint8), 60)])
    if invert:
        bits = 1 - bits
    soft = np.where(bits == 1, soft_hi, soft_lo).astype(np.int16)
    return np.concatenate([np.array([-1], dtype=np.int16), soft])
