"""CPU checks of the channelizer's rational rates (output_rate / input_rate = L/M): the library's ratio rule, the prototype
design at L * input_rate against scipy and its specification, and the float64 polyphase statement (tests/chan_poly_ref.py)
against tests/chan_ref.py at L = 1 and against zero-stuff, filter and keep-every-M at L > 1."""
import ctypes

import numpy as np
import pytest
from scipy import signal

from chan_poly_ref import chan_poly_ref, n_outputs
from chan_ref import TWO32, chan_ref, llround
from conftest import has_cuda

RATIOS = {2.048e6: (3, 128), 1.024e6: (3, 64), 2.5e6: (12, 625), 3e6: (2, 125), 10e6: (3, 625), 2.4e6: (1, 50)}
RATES = [2.048e6, 2.5e6, 1.024e6]
PASSBANDS = [12000.0, 3000.0, 10000.0]
EXPECTED_T_TP = {2.048e6: [(1859, 620), (1063, 355), (1593, 531)],
                 2.5e6: [(9065, 756), (5181, 432), (7771, 648)],
                 1.024e6: [(931, 311), (533, 178), (797, 266)]}


def _jb():
    import jaero_b200
    return jaero_b200


def _scipy_design(input_rate, L, passband_hz, audio_hz=12000.0, output_rate=48000.0):
    fp = passband_hz / 2
    fs = min(2 * audio_hz, output_rate - 2 * audio_hz) - fp
    T, beta = signal.kaiserord(60.0, (fs - fp) / (L * input_rate / 2))
    T |= 1
    return L * signal.firwin(T, (fp + fs) / 2, window=("kaiser", beta), fs=L * input_rate), fp, fs


def test_ratios_follow_the_library_rule():
    jb = _jb()
    L = jb.lib()
    for rate, want in RATIOS.items():
        assert jb.channelizer_ratio(rate) == want, rate
        s = jb.ChanSettings(0, 0, rate, 48000.0, 12000.0, 12000.0, 1.0)
        lo, mo = ctypes.c_int(), ctypes.c_int()
        assert L.jaero_chan_ratio(ctypes.byref(s), ctypes.byref(lo), ctypes.byref(mo)) == 0
        assert (lo.value, mo.value) == want
    assert jb.channelizer_ratio(3e6, output_rate=24000.0, audio_hz=6000.0, passband_hz=3000.0) == (1, 125)
    for rate, pb in ((72000.0, 12000.0), (80000.0, 12000.0), (2.4e6 + 1, 12000.0), (10e6, 23900.0)):
        s = jb.ChanSettings(0, 0, rate, 48000.0, 12000.0, pb, 1.0)
        assert L.jaero_chan_ratio(ctypes.byref(s), None, None) == -1, rate
        assert L.jaero_chan_taps(ctypes.byref(s), None, 0) == -1, rate
        with pytest.raises(jb.JaeroError):
            jb.channelizer_ratio(rate, passband_hz=pb)
    with pytest.raises(jb.JaeroError, match="L/M with L <= 64 and M >= 2L"):
        jb.channelizer_ratio(80000.0)
    with pytest.raises(jb.JaeroError, match="8191 taps per phase"):
        jb.channelizer_ratio(10e6, passband_hz=23900.0)


@pytest.mark.parametrize("input_rate", RATES)
def test_prototype_equals_scipy_at_l_times_input_rate(input_rate):
    jb = _jb()
    L, _ = RATIOS[input_rate]
    got_sizes = []
    for pb in PASSBANDS:
        want, _, _ = _scipy_design(input_rate, L, pb)
        got = jb.channelizer_taps(input_rate, passband_hz=pb)
        assert len(got) == len(want) and len(got) % 2 == 1
        assert np.max(np.abs(got - want)) <= 1e-12 * np.max(np.abs(want)), (input_rate, pb)
        assert abs(got.sum() - L) < 1e-12 * L
        got_sizes.append((len(got), -(-len(got) // L)))
    assert got_sizes == EXPECTED_T_TP[input_rate]


@pytest.mark.parametrize("input_rate", RATES)
def test_prototype_meets_passband_and_stopband(input_rate):
    jb = _jb()
    L, _ = RATIOS[input_rate]
    for pb in PASSBANDS:
        h = jb.channelizer_taps(input_rate, passband_hz=pb) / L
        _, fp, fs = _scipy_design(input_rate, L, pb)
        f, H = signal.freqz(h, worN=np.linspace(0.0, 60000.0, 1 << 16), fs=L * input_rate)
        db = 20 * np.log10(np.maximum(np.abs(H), 1e-300))
        assert np.all(np.abs(db[f <= fp]) <= 0.05), (input_rate, pb, db[f <= fp].min())
        floor = -58.0 if pb >= 10000.0 else -57.5
        assert np.all(db[f >= fs] <= floor), (input_rate, pb, db[f >= fs].max())
        # the fine grid above covers the band edges; the rest of the stopband, up to L * input_rate / 2, on a coarser one
        f2, H2 = signal.freqz(h, worN=1 << 18, fs=L * input_rate)
        assert 20 * np.log10(np.abs(H2[f2 >= fs]).max()) <= floor, (input_rate, pb)


def _tones(n, fs, seed):
    rng = np.random.default_rng(seed)
    t = np.arange(n)
    x = rng.normal(0, 2000.0, n) + 1j * rng.normal(0, 2000.0, n)
    for f in rng.uniform(-0.45 * fs, 0.45 * fs, 4):
        x += 6000.0 * np.exp(2j * np.pi * (f * t / fs + rng.uniform()))
    return x


def test_poly_ref_equals_chan_ref_at_integer_rates():
    jb = _jb()
    for fs, pb in ((2.4e6, 12000.0), (1.536e6, 3000.0)):
        L, M = jb.channelizer_ratio(fs, passband_hz=pb)
        assert L == 1
        h = jb.channelizer_taps(fs, passband_hz=pb)
        x = np.rint(_tones(300 * M + 7, fs, 3))
        off = [0.0, -301234.5, 456789.25]
        want = chan_ref(x, h, off, fs, gain=0.7)
        got = chan_poly_ref(x, h, L, M, off, fs, gain=0.7)
        assert got.shape == want.shape and np.array_equal(got, want)


@pytest.mark.parametrize("input_rate", [2.048e6, 2.5e6])
def test_poly_ref_equals_zero_stuff_filter_decimate(input_rate):
    """a_c[m] = (h * u)[mM] with u the mixed input zero-stuffed by L: u[iL] = x[i] e^{-2 pi j phi_c(i)/2^32}."""
    jb = _jb()
    L, M = jb.channelizer_ratio(input_rate)
    assert L in (3, 12)
    h = jb.channelizer_taps(input_rate)
    N = 20 * M + 5
    x = _tones(N, input_rate, L)
    off = [-345678.9, 0.0, 512345.25]
    a = chan_poly_ref(x, h, L, M, off, input_rate, pre_rounding=True)
    n_out = n_outputs(N, L, M)
    assert a.shape == (3, n_out)
    for c, o in enumerate(off):
        inc = llround(o / input_rate * TWO32) % TWO32
        phi = (np.arange(N, dtype=np.uint64) * np.uint64(inc)) % np.uint64(TWO32)
        u = np.zeros(N * L, dtype=np.complex128)
        u[::L] = x * np.exp(-2j * np.pi * phi.astype(np.float64) / TWO32)
        y = np.convolve(u, h)[: N * L]
        want = y[np.arange(n_out) * M]
        assert np.max(np.abs(a[c] - want)) <= 1e-9 * np.max(np.abs(want)), (input_rate, o)
        assert (n_out - 1) * M < N * L <= n_out * M                         # every output with n_m inside x, no more


@pytest.mark.skipif(has_cuda(), reason="only meaningful on a box without a GPU")
def test_rational_channelizer_has_no_cpu_fallback():
    jb = _jb()
    with pytest.raises(jb.JaeroError, match="no such CUDA device"):
        jb.Channelizer([0.0, 25000.0], 2.048e6, iq_format="cu8")
