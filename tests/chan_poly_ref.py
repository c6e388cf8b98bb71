"""float64 statement of the channelizer's rational-rate definition (include/jaero_b200.h, "device channelizer"), written out
literally: output m sits at input time mM/L, n_m = floor(mM/L), p_m = mM mod L; mix each channel to 0 Hz with the uint32
phase phi_c(n), sum h[kL + p_m] x[n_m - k] over the Tp = ceil(T/L) taps of branch p_m (x[n<0] = 0, h[j >= T] = 0), rotate by
psi(m), scale, round half to even, saturate. With L = 1 it is tests/chan_ref.py."""
import numpy as np

from chan_ref import TWO32, llround


def n_outputs(n_in, L, M):
    """outputs with n_m inside the first n_in input samples: ceil(L n_in / M)"""
    return (L * n_in + M - 1) // M


def chan_poly_ref(x, h, L, M, offsets_hz, input_rate, output_rate=48000.0, audio_hz=12000.0, gain=1.0, n_out=None,
                  block=2048, pre_rounding=False):
    """x: complex128 input from sample 0; h: the prototype (length T, sum L). Returns int16 [C, n_out], or the complex128
    a_c[m] before the rotation when pre_rounding is set. n_out defaults to every m with n_m inside x."""
    T = len(h)
    Tp = (T + L - 1) // L
    N = len(x)
    n_out = n_outputs(N, L, M) if n_out is None else n_out
    hp = np.zeros(Tp * L)
    hp[:T] = h
    branch = hp.reshape(Tp, L).T                                             # branch[p, k] = h[kL + p]
    m = np.arange(n_out, dtype=np.int64)
    n_m = (m * M) // L
    p_m = (m * M) % L
    inc_a = llround(audio_hz / output_rate * TWO32) % TWO32
    psi = (m.astype(np.uint64) * np.uint64(inc_a)) % np.uint64(TWO32)
    rot = np.exp(2j * np.pi * psi.astype(np.float64) / TWO32)
    xp = np.concatenate([np.zeros(Tp - 1, dtype=np.complex128), x])           # xp[Tp-1+n] = x[n]
    n = np.arange(-(Tp - 1), N, dtype=np.int64)
    out = np.empty((len(offsets_hz), n_out), dtype=np.complex128 if pre_rounding else np.int16)
    for c, off in enumerate(offsets_hz):
        inc = llround(off / input_rate * TWO32) % TWO32
        phi = (n.astype(np.uint64) * np.uint64(inc)) % np.uint64(TWO32)       # n < 0 wraps too, but x is 0 there
        mixed = xp * np.exp(-2j * np.pi * phi.astype(np.float64) / TWO32)
        a = np.empty(n_out, dtype=np.complex128)
        for b0 in range(0, n_out, block):
            mm = np.arange(b0, min(n_out, b0 + block))
            idx = (Tp - 1) + n_m[mm][:, None] - np.arange(Tp)[None, :]        # x[n_m - k]
            for p in range(L):
                sel = p_m[mm] == p
                a[mm[sel]] = mixed[idx[sel]] @ branch[p]
        if pre_rounding:
            out[c] = a
        else:
            v = np.rint(gain * np.real(a * rot))
            out[c] = np.clip(v, -32768, 32767).astype(np.int16)
    return out
