"""CPU checks of the device channelizer's host side: the filter design equals scipy's Kaiser design and meets its
specification, every invalid setting is rejected before a device is touched, the C struct matches its ctypes mirror, and
the float64 reference (tests/chan_ref.py) agrees with the closed form on a pure tone."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
from scipy import signal

from chan_ref import TWO32, chan_ref, llround
from conftest import ROOT, has_cuda

RATES = [1.536e6, 2.4e6, 6e6]
DESIGNS = [(12000.0, 12000.0), (12000.0, 3000.0), (12000.0, 10000.0), (8000.0, 8000.0), (6000.0, 2400.0)]
# the issue's table: audio 12 kHz, output 48 kHz, passband 12 000 / 3000 / 10 000 Hz
EXPECTED_T = {1.536e6: (467, 267, 399), 2.4e6: (727, 417, 623), 6e6: (1815, 1037, 1555)}


def _L():
    import jaero_b200
    return jaero_b200, jaero_b200.lib()


def _settings(jb, input_rate=2.4e6, output_rate=48000.0, audio_hz=12000.0, passband_hz=12000.0, iq_format=0, gain=1.0):
    return jb.ChanSettings(iq_format, 0, input_rate, output_rate, audio_hz, passband_hz, gain)


def _scipy_design(input_rate, audio_hz, passband_hz, output_rate=48000.0):
    fp = passband_hz / 2
    fs = min(2 * audio_hz, output_rate - 2 * audio_hz) - fp
    T, beta = signal.kaiserord(60.0, (fs - fp) / (input_rate / 2))
    T |= 1
    return signal.firwin(T, (fp + fs) / 2, window=("kaiser", beta), fs=input_rate), fp, fs


@pytest.mark.parametrize("input_rate", RATES)
def test_taps_equal_scipy_kaiser_design(input_rate):
    jb, _ = _L()
    for audio, pb in DESIGNS:
        want, _, _ = _scipy_design(input_rate, audio, pb)
        got = jb.channelizer_taps(input_rate, audio_hz=audio, passband_hz=pb)
        assert len(got) == len(want) and len(got) % 2 == 1
        assert np.max(np.abs(got - want)) <= 1e-12 * np.max(np.abs(want)), (input_rate, audio, pb)
        assert abs(got.sum() - 1.0) < 1e-12
    assert tuple(len(jb.channelizer_taps(input_rate, passband_hz=pb)) for pb in (12000.0, 3000.0, 10000.0)) == EXPECTED_T[input_rate]


@pytest.mark.parametrize("input_rate", RATES)
def test_taps_meet_passband_and_stopband(input_rate):
    """Ripple within +-0.05 dB for f <= f_p. Kaiser's length estimate for A = 60 dB is approximate: the designs here reach
    57.6 dB (widest relative transition, the 3 kHz MSK passband) to 59.9 dB, so the bound checked is 57.5 dB, and 58 dB
    for the 10 and 12 kHz passbands."""
    jb, _ = _L()
    for audio, pb in DESIGNS:
        h = jb.channelizer_taps(input_rate, audio_hz=audio, passband_hz=pb)
        _, fp, fs = _scipy_design(input_rate, audio, pb)
        f, H = signal.freqz(h, worN=1 << 19, fs=input_rate)
        db = 20 * np.log10(np.maximum(np.abs(H), 1e-300))
        assert np.all(np.abs(db[f <= fp]) <= 0.05), (input_rate, audio, pb, db[f <= fp].min(), db[f <= fp].max())
        floor = -58.0 if pb >= 10000.0 else -57.5
        assert np.all(db[f >= fs] <= floor), (input_rate, audio, pb, db[f >= fs].max())


def test_invalid_settings_are_rejected_before_any_device():
    jb, L = _L()
    bad = [
        dict(iq_format=2), dict(iq_format=-1),
        dict(input_rate=2.4e6 + 1), dict(output_rate=48000.0, input_rate=48000.0), dict(input_rate=72000.0),
        dict(input_rate=-2.4e6), dict(output_rate=0.0), dict(input_rate=float("nan")),
        dict(audio_hz=0.0), dict(audio_hz=-100.0), dict(audio_hz=24000.0), dict(audio_hz=30000.0),
        dict(passband_hz=24000.0), dict(audio_hz=3000.0, passband_hz=12000.0), dict(passband_hz=0.0),
        dict(input_rate=48000.0 * 200, audio_hz=12000.0, passband_hz=23900.0),       # T > 8191
        dict(gain=0.0), dict(gain=-1.0), dict(gain=float("inf")), dict(gain=float("nan")),
    ]
    for kw in bad:
        s = _settings(jb, **kw)
        assert L.jaero_chan_taps(ctypes.byref(s), None, 0) == -1, kw
        h = ctypes.c_void_p()
        off = np.zeros(4)
        assert L.jaero_chan_create(ctypes.byref(s), 4, jb._p(off), 0, ctypes.byref(h)) == -1, kw
        assert not h.value
    s = _settings(jb)
    assert L.jaero_chan_taps(ctypes.byref(s), None, 0) == 727
    h = ctypes.c_void_p()
    for off in ([1.2e6 - 5999.0], [-1.2e6 + 5999.0], [float("nan")]):            # |offset| + passband/2 > input_rate/2
        o = np.array(off)
        assert L.jaero_chan_create(ctypes.byref(s), 1, jb._p(o), 0, ctypes.byref(h)) == -1
    o = np.zeros(1)
    for n in (0, -3):
        assert L.jaero_chan_create(ctypes.byref(s), n, jb._p(o), 0, ctypes.byref(h)) == -1
    assert L.jaero_chan_create(None, 1, jb._p(o), 0, ctypes.byref(h)) == -1
    with pytest.raises(jb.JaeroError):
        jb.channelizer_taps(2.4e6, iq_format="cf32")


def test_chan_settings_layout_matches_header(tmp_path):
    jb, _ = _L()
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "jaero_b200.h"\nint main(void){printf("%zu %zu %zu %zu %zu %zu %zu\\n",'
                   'sizeof(jaero_chan_settings), offsetof(jaero_chan_settings, reserved), offsetof(jaero_chan_settings, input_rate),'
                   'offsetof(jaero_chan_settings, output_rate), offsetof(jaero_chan_settings, audio_hz),'
                   'offsetof(jaero_chan_settings, passband_hz), offsetof(jaero_chan_settings, gain));return 0;}\n')
    exe = str(tmp_path / "layout")
    subprocess.run(["gcc", "-I" + os.path.join(ROOT, "include"), str(src), "-o", exe], check=True)
    got = [int(x) for x in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split()]
    S = jb.ChanSettings
    assert got == [ctypes.sizeof(S), S.reserved.offset, S.input_rate.offset, S.output_rate.offset, S.audio_hz.offset,
                   S.passband_hz.offset, S.gain.offset]


@pytest.mark.skipif(has_cuda(), reason="only meaningful on a box without a GPU")
def test_channelizer_has_no_cpu_fallback():
    jb, _ = _L()
    with pytest.raises(jb.JaeroError, match="no such CUDA device"):
        jb.Channelizer([0.0, 25000.0], 2.4e6)


def test_chan_ref_tone_matches_closed_form():
    """x[n] = A e^{2 pi j f n / Fs}: a_c[m] = A e^{2 pi j nu m D} sum_k h[k] e^{-2 pi j nu k} once the filter is full,
    with nu = f / Fs - inc_c / 2^32."""
    jb, _ = _L()
    Fs, D = 1.536e6, 32
    h = jb.channelizer_taps(Fs)
    off, f, A, gain = -301234.5, -301234.5 + 2345.0, 9000.0, 1.5
    N = 40000
    x = A * np.exp(2j * np.pi * f * np.arange(N) / Fs)
    got = chan_ref(x, h, [off], Fs, gain=gain)[0]
    inc = llround(off / Fs * TWO32) % TWO32
    nu = f / Fs - inc / TWO32
    Hnu = np.sum(h * np.exp(-2j * np.pi * nu * np.arange(len(h))))
    m = np.arange(len(got))
    psi = (m.astype(np.uint64) * np.uint64(llround(12000.0 / 48000.0 * TWO32) % TWO32)) % np.uint64(TWO32)
    want = gain * np.real(A * np.exp(2j * np.pi * nu * m * D) * Hnu * np.exp(2j * np.pi * psi.astype(np.float64) / TWO32))
    full = m * D >= len(h) - 1
    assert full.sum() > 1000
    d = np.abs(got[full].astype(np.float64) - want[full])
    assert d.max() <= 0.5 + 1e-6
    assert np.abs(got[full] - np.rint(want[full])).max() <= 1
    assert np.mean(got[full] == np.rint(want[full])) >= 0.999
