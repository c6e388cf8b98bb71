"""float64 statement of the channelizer's definition (include/jaero_b200.h, "device channelizer"), written out literally:
mix each channel to 0 Hz with the uint32 phase phi_c(n), convolve with h at the decimated points (direct sum, x[n<0] = 0),
rotate by psi(m), scale, round half to even, saturate."""
import numpy as np

TWO32 = 4294967296


def llround(v):
    return int(np.sign(v) * np.floor(abs(v) + 0.5))


def iq_to_complex(iq, iq_format):
    """[n, 2] int16 (cs16) or uint8 (cu8) -> complex128 x[n]"""
    a = np.asarray(iq).astype(np.float64)
    if iq_format == "cu8":
        a = (a - 127.5) * 256.0
    return a[:, 0] + 1j * a[:, 1]


def chan_ref(x, h, offsets_hz, input_rate, output_rate=48000.0, audio_hz=12000.0, gain=1.0, n_out=None, block=4096):
    """x: complex128 input from sample 0; returns int16 [C, M] with M = every m whose mD lies inside x (or n_out)."""
    D = int(round(input_rate / output_rate))
    T = len(h)
    N = len(x)
    M = (N + D - 1) // D if n_out is None else n_out
    inc_a = llround(audio_hz / output_rate * TWO32) % TWO32
    m = np.arange(M, dtype=np.uint64)
    psi = (m * np.uint64(inc_a)) % np.uint64(TWO32)
    rot = np.exp(2j * np.pi * psi.astype(np.float64) / TWO32)
    xp = np.concatenate([np.zeros(T - 1, dtype=np.complex128), x])            # xp[T-1+n] = x[n]
    n = np.arange(-(T - 1), N, dtype=np.int64)
    out = np.empty((len(offsets_hz), M), dtype=np.int16)
    for c, off in enumerate(offsets_hz):
        inc = llround(off / input_rate * TWO32) % TWO32
        phi = (n.astype(np.uint64) * np.uint64(inc)) % np.uint64(TWO32)       # n < 0 wraps too, but x is 0 there
        mixed = xp * np.exp(-2j * np.pi * phi.astype(np.float64) / TWO32)
        a = np.empty(M, dtype=np.complex128)
        for b0 in range(0, M, block):
            mm = np.arange(b0, min(M, b0 + block))
            idx = (T - 1) + mm[:, None] * D - np.arange(T)[None, :]          # x[mD - k]
            a[mm] = mixed[idx] @ h
        v = np.rint(gain * np.real(a * rot))
        out[c] = np.clip(v, -32768, 32767).astype(np.int16)
    return out
