"""CPU pins of the host design module (jaero_b200/csrc/host_design.cpp): what every create call derives from its settings
before it touches a device. The demodulator kernels reproduce the reference bit for bit only with exactly these values, so
they are compared with the reference's stored results where the reference has them (RRC taps, trig tables, scrambler) and
otherwise with digests of the values the product computed before the design math moved into this module. Also: with no
device present, every unsupported setting is reported as a bad argument, not as a missing device."""
import hashlib
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, has_cuda
from ref_pins import same

CSRC = os.path.join(ROOT, "jaero_b200", "csrc")

# sha256 of `host_design_driver plan <mode>` / `pchannel <fb>` / `rt <fb>`, recorded from the create calls of the
# library as it was before the design module existed (its capi.cu run on the host against a CUDA runtime stand-in)
PLAN_DIGESTS = {
    "plan oqpsk10500": "bfe034705a9c559cd6a45892390b28d19778a82eb13cf99d3af50319db61bfce",
    "plan oqpsk8400": "5c2e0410e5bbd45052557b0a99e11626a182b294167c40254196cbd4475afce4",
    "plan msk600": "9a0678928740dba70ab72f35273e92cf6f7fe1f8d11b7cdb371d6e9112d2dfe3",
    "plan msk1200": "88eea3d31d7e53ca0618c47d4539d3d4512310cd8909f39157bc11fec1046783",
    "plan burst_msk600": "0b1e8ebc70fec78ec9ec6e5dbf160222d3d9328ddef68d9181100fcb90e5cab6",
    "plan burst_msk1200": "5ffbab9e64bcd869de3053d5b100607a12aca64bc419833a4af536dda460e362",
    "plan burst_oqpsk10500": "0c04f1c256778f9da3080e24c7a4dfca410bc0ff708830c263c746d8fc1ab66a",
    "pchannel 600": "f9d3656015ab78ad408edbb8344afa8c408e54d29dbad7bc462097e1d21d1741",
    "pchannel 1200": "dc1a0b995daee55d15b228d5b9ce6a62b8ee6c11219b7736802432c190db688b",
    "pchannel 10500": "7204e2ea9072bfa2138ae34841cbe8c86ea27d4600ff9d00569fcd8dbf40d6e2",
    "rt 600": "339360d76549f23d056d96c66a938861c4e427895e30c0966a88edd5d805d524",
    "rt 1200": "13c4c8f226f3f86e32047985facf47731641160e5f41daec2523ed813eddc4b0",
    "rt 10500": "21e395dcef7b3dca0b84ca196afac3292dfe72e6a5955ca89fdcf177cd8b8ceb",
}


@pytest.fixture(scope="module")
def driver(tmp_path_factory):
    """tests/cpp/host_design_driver.cpp + host_design.cpp, compiled with the host flags jaero_b200/build.py gives nvcc"""
    from jaero_b200 import build
    cuda_inc = os.path.join(os.path.dirname(os.path.dirname(build.NVCC)), "include")
    exe = str(tmp_path_factory.mktemp("hd") / "host_design_driver")
    cmd = ["g++", "-O3", "-std=c++17", "-fPIC", "-fno-fast-math", "-I" + cuda_inc, os.path.join(ROOT, "tests", "cpp", "host_design_driver.cpp"),
           os.path.join(CSRC, "host_design.cpp"), "-o", exe]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return exe


def _run(exe, *args):
    r = subprocess.run([exe] + list(args), capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    return r.stdout


def _values(text):
    """the numbers of a dump_v block: header line `name n`, then n values"""
    lines = text.split("\n")
    out, i = {}, 0
    while i < len(lines) and lines[i]:
        name, n = lines[i].split()
        out[name] = np.array([float(v) for v in lines[i + 1:i + 1 + int(n)]])
        i += 1 + int(n)
    return out


def _no_recording():
    raise AssertionError("the reference's result is stored in tests/golden/ref_pins.json")


def test_rrc_taps_trig_tables_and_scrambler_equal_the_reference(driver):
    taps = _values(_run(driver, "rrc"))["rrc"]
    padded = np.zeros(64)
    padded[:len(taps)] = taps
    assert len(taps) == 55 and same([55, padded], "oracle/rrc_taps", _no_recording)
    t = _values(_run(driver, "trig"))
    assert same([t["sin"], t["cos"]], "oracle/trig_tables", _no_recording)
    seq = np.array([int(v) for v in _run(driver, "scrambler").split()], dtype=np.int32)
    assert same(seq, "fec/scrambler", _no_recording)


@pytest.mark.parametrize("args", sorted(PLAN_DIGESTS))
def test_create_plans_are_unchanged(driver, args):
    """taps, delay weights, pre-filter / Hilbert spectra, estimator twiddles and window, and every scalar parameter"""
    text = _run(driver, *args.split())
    assert hashlib.sha256(text.encode()).hexdigest() == PLAN_DIGESTS[args], text[:2000]


@pytest.mark.skipif(has_cuda(), reason="checks the order of validation and device selection on a machine without a GPU")
def test_bad_settings_are_argument_errors_even_without_a_device():
    """the cases of test_gpu_boundary.py::test_every_create_error_branch_returns_an_error, through the real library: each
    create validates its settings before it looks for a device"""
    import ctypes
    import jaero_b200 as jb
    L = jb.lib()
    OQ, MSK = jb.KIND_OQPSK, jb.KIND_MSK

    def batch(kind, n, fb, Fs, power=14):
        s = jb.Settings(kind, power, 8000.0, 10500.0, float(fb), float(Fs), 0.65, 0, 0, 0, 1)
        h = ctypes.c_void_p()
        return L.jaero_batch_create(ctypes.byref(s), n, None, 0, ctypes.byref(h)), L.jaero_last_error().decode()

    for case in [(OQ, 2, 10500, 44100), (OQ, 2, 10500, 48001), (OQ, 2, 10500, 192000), (MSK, 2, 100, 48000, 13), (MSK, 2, 600, 48010, 13),
                 (OQ, 0, 10500, 48000), (OQ, 2, 10500, 48000, 9), (OQ, 2, -1, 48000), (7, 2, 10500, 48000)]:
        rc, msg = batch(*case)
        assert rc == -1 and msg and "device" not in msg, (case, rc, msg)
    for make in [lambda: jb.BurstMskBatch(2, fb=1200, Fs=44100), lambda: jb.BurstMskBatch(2, fb=300), lambda: jb.BurstOqpskBatch(2, fb=8400),
                 lambda: jb.PChannelBatch(2, 8400), lambda: jb.RTChannelBatch(2, 8400), lambda: jb.ViterbiBatch(2, 23)]:
        with pytest.raises(jb.JaeroError, match=r"error -1: "):
            make()
    rc, msg = batch(OQ, 2, 10500, 48000)                     # a valid create reaches the device check
    assert rc == -2 and "no such CUDA device" in msg, msg
