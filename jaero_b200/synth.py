"""Synthetic Inmarsat-Aero P-channel transmit chain (test / bench signal source).

The reference has no modulator; this inverts AeroL::Decode (JAERO/aerol.cpp:1124-1322,1540-1610,
1990-2039) and the demodulators' conventions (SURVEY.md App. D): 12-byte signal units with CRC-16
(aerol.h:334-362) -> LSB-first bits -> scrambler (aerol.h:397-419) -> K=7 r=1/2 encoder, polys
109/79, continuous across frames -> 64xN block interleaver (aerol.cpp:550-566) -> frame = UW +
header (+178 dummy bits at 10.5k) + data -> OQPSK (RRC alpha=1, 5250 Bd per arm, arms offset by
one bit) or MSK -> real passband int16 at Fs = 48 kHz.

Pure numpy; the heavy per-channel replication for the bench is done with torch on the GPU in bench.py.
"""
import numpy as np

UW = 0xE15AE893                      # aerol.cpp:947


def crc16(data):
    """AeroLcrc16::calcusingbytes (aerol.h:334-362): reflected 0x8408, init 0xFFFF, final complement."""
    crc = 0xFFFF
    for byte in data:
        b = int(byte)
        for _ in range(8):
            mb = b & 1
            b >>= 1
            cb = crc & 1
            crc >>= 1
            if cb ^ mb:
                crc ^= 0x8408
    return (~crc) & 0xFFFF


def make_su(rng, kind=None):
    """One 12-byte signal unit: 10 payload bytes + CRC (low byte first, aerol.cpp:1591-1592)."""
    body = rng.integers(0, 256, size=10, dtype=np.uint8)
    if kind is not None:
        body[0] = kind
    c = crc16(body)
    return np.concatenate([body, np.array([c & 0xFF, c >> 8], dtype=np.uint8)])


def scrambler_sequence(n):
    """AeroLScrambler (aerol.h:397-419)."""
    st = [1, 1, 0, 1, 0, 0, 1, 0, 1, 0, 1, 1, 0, 0, 1]
    out = np.zeros(n, dtype=np.uint8)
    for a in range(n):
        v = st[0] ^ st[14]
        out[a] = v
        st = [v] + st[:-1]
    return out


def conv_encode_stream(bits, state=0):
    """libcorrect convention: sr=(sr<<1|bit)&127, outputs parity(sr&109) then parity(sr&79)."""
    out = np.zeros(2 * len(bits), dtype=np.uint8)
    sr = state
    p109 = np.array([bin(i & 109).count("1") & 1 for i in range(128)], dtype=np.uint8)
    p79 = np.array([bin(i & 79).count("1") & 1 for i in range(128)], dtype=np.uint8)
    for k, b in enumerate(bits):
        sr = ((sr << 1) | int(b)) & 127
        out[2 * k] = p109[sr]
        out[2 * k + 1] = p79[sr]
    return out, sr


def interleave(coded, cols):
    """Inverse of AeroLInterleaver::deinterleave_ba: coded bit k=j*64+i goes to ((i*27)%64)*cols + j."""
    n = 64 * cols
    assert len(coded) == n
    k = np.arange(n)
    i = k % 64
    j = k // 64
    out = np.zeros(n, dtype=np.uint8)
    out[((i * 27) % 64) * cols + j] = coded
    return out


def frame_params(fb):
    fb = int(fb)
    if fb == 10500:
        return dict(cols=78, blocks=1, header_extra=178, uw_interleaved=True, sus=26, frame_bits=5250)
    if fb == 1200:
        return dict(cols=9, blocks=2, header_extra=0, uw_interleaved=False, sus=12, frame_bits=1200)
    if fb == 600:
        return dict(cols=6, blocks=3, header_extra=0, uw_interleaved=False, sus=12, frame_bits=1200)
    raise ValueError("unsupported P-channel rate")


def pchannel_bits(fb, n_frames, seed=0, return_sus=False, loop=False, even_parity=False):
    """Serial channel bits for n_frames P-channel frames (and the signal units they carry).
    loop=True: the convolutional encoder starts in the state it ends in (tail-biting), so the frame sequence can be
    repeated for ever without a decoding glitch at the seam. even_parity=True: the whole bit sequence is given even parity
    (needed to close a differentially pre-coded MSK waveform on itself) by setting the super-frame marker of the last frame's
    header when necessary - with a tail-biting rate-1/2 code of two odd-weight polynomials the coded bits always have even
    parity, so only the 16 header bits decide."""
    fp = frame_params(fb)
    rng = np.random.default_rng(seed)
    uw_bits = np.array([(UW >> (31 - i)) & 1 for i in range(32)], dtype=np.uint8)
    info_bits_per_frame = fp["blocks"] * 64 * fp["cols"] // 2
    n_sus = info_bits_per_frame // 96
    scr = scrambler_sequence(info_bits_per_frame)
    out = _pchannel_bits_once(fp, rng, n_frames, uw_bits, n_sus, scr, loop, even_parity)
    return out if return_sus else out[0]


def _pchannel_bits_once(fp, rng, n_frames, uw_bits, n_sus, scr, loop, even_parity=False):
    payloads, all_sus, dummies = [], [], []
    for f in range(n_frames):
        sus = [make_su(rng, 0x01 if (k % 3) else None) for k in range(n_sus)]
        all_sus.append(np.stack(sus))
        payloads.append(np.unpackbits(np.concatenate(sus), bitorder="little") ^ scr)   # LSB-first (aerol.cpp:1568-1580); the
        #                                                           scrambler restarts every frame (:2010,2015)
        dummies.append(rng.integers(0, 2, size=fp["header_extra"], dtype=np.uint8))
    enc_state = 0
    if loop:                                                      # encoder state after the last frame = its last 7 input bits
        for b in payloads[-1][-7:]:
            enc_state = ((enc_state << 1) | int(b)) & 127
    frames, headers_at = [], []
    for f in range(n_frames):
        bits = payloads[f]
        coded, enc_state = conv_encode_stream(bits, enc_state)
        blocks = [interleave(coded[b * 64 * fp["cols"]:(b + 1) * 64 * fp["cols"]], fp["cols"]) for b in range(fp["blocks"])]
        # formatid(4) = 1 | supfrmaker(4) | framecounter1(4) | framecounter2(4)  (aerol.cpp:1275-1319)
        header = np.array([(0x1000 | ((f & 15) << 4) | (f & 15)) >> (15 - i) & 1 for i in range(16)], dtype=np.uint8)
        headers_at.append(sum(len(x) for x in frames) + len(uw_bits) * (2 if fp["uw_interleaved"] else 1))
        if fp["uw_interleaved"]:
            uw = np.repeat(uw_bits, 2)                            # same word on both arms (aerol.cpp:959-960)
        else:
            uw = uw_bits
        frame = np.concatenate([uw, header, dummies[f]] + blocks)
        assert len(frame) == fp["frame_bits"], (len(frame), fp["frame_bits"])
        frames.append(frame)
    allbits = np.concatenate(frames)
    if even_parity and (int(allbits.sum()) & 1):
        allbits[headers_at[-1] + 7] ^= 1                          # last frame: supfrmaker 0 -> 1
    return allbits, np.stack(all_sus)


def rrc_pulse(alpha, span_symbols, sps):
    """Root-raised-cosine pulse sampled at `sps` samples/symbol (closed form as DSP.h:316-338)."""
    n = int(round(span_symbols * sps))
    if n % 2 == 0:
        n += 1
    t = (np.arange(n) - (n - 1) / 2.0) / sps
    h = np.zeros(n)
    for i, ti in enumerate(t):
        if abs(ti) < 1e-12:
            h[i] = 1.0 - alpha + 4 * alpha / np.pi
        elif abs(abs(4 * alpha * ti) - 1.0) < 1e-9:
            h[i] = alpha / np.sqrt(2) * ((1 + 2 / np.pi) * np.sin(np.pi / (4 * alpha)) + (1 - 2 / np.pi) * np.cos(np.pi / (4 * alpha)))
        else:
            h[i] = (np.sin(np.pi * ti * (1 - alpha)) + 4 * alpha * ti * np.cos(np.pi * ti * (1 + alpha))) / (np.pi * ti * (1 - (4 * alpha * ti) ** 2))
    return h / np.sqrt(np.sum(h ** 2) / sps)


def oqpsk_envelope(bits, fb, Fs=48000.0, alpha=1.0):
    """Complex envelope of the OQPSK signal (circular, i.e. seamless when looped). Serial bit n sits in
    half-symbol slot n (duration 1/fb): even bits drive the quadrature arm, odd bits the in-phase arm one
    slot later — the order in which the demodulator emits them (pt_d.imag then pt.real,
    oqpskdemodulator.cpp:503,569-579). Pulse: root-raised-cosine, symbol rate fb/2 per arm."""
    from fractions import Fraction
    n_bits = len(bits)
    fr = Fraction(int(Fs), int(fb))               # samples per bit slot, e.g. 32/7
    up, spb_up = fr.denominator, fr.numerator     # work on a grid of Fs*up where a slot is spb_up samples
    assert (n_bits * spb_up) % up == 0, "whole number of output samples required"
    n_up = n_bits * spb_up
    sym = 2.0 * bits.astype(np.float64) - 1.0
    xq = np.zeros(n_up); xi = np.zeros(n_up)
    xq[(np.arange(0, n_bits, 2) * spb_up)] = sym[0::2]
    xi[(np.arange(1, n_bits, 2) * spb_up)] = sym[1::2]
    freqs = np.abs(np.fft.fftfreq(n_up, d=1.0 / (Fs * up)))
    Rs = fb / 2.0
    f1, f2 = (1 - alpha) * Rs / 2, (1 + alpha) * Rs / 2
    H = np.zeros(n_up)
    H[freqs <= f1] = 1.0
    m = (freqs > f1) & (freqs <= f2)
    H[m] = np.sqrt(0.5 * (1 + np.cos(np.pi / (alpha * Rs) * (freqs[m] - f1))))
    q = np.fft.ifft(np.fft.fft(xq) * H).real[::up]
    i = np.fft.ifft(np.fft.fft(xi) * H).real[::up]
    env = i + 1j * q
    return env / np.sqrt(np.mean(np.abs(env) ** 2))


def to_passband_int16(env, fc, Fs=48000.0, ebn0_db=None, fb=10500.0, rms=0.2, phase=0.0, rng=None, delay=0):
    """Real passband x[n] = Re{env[n] e^{j(2 pi fc n/Fs + phase)}} + AWGN, scaled to `rms` of full scale."""
    n = np.arange(len(env))
    if delay:
        env = np.roll(env, delay)
    x = np.real(env * np.exp(1j * (2 * np.pi * fc * n / Fs + phase)))       # power 1/2 for unit-power env
    if ebn0_db is not None:
        rng = rng or np.random.default_rng(0)
        # Eb = P_signal * (Fs/fb) samples ; N0/2 per real sample = sigma^2
        ps = np.mean(x ** 2)
        eb = ps * Fs / fb
        n0 = eb / (10 ** (ebn0_db / 10.0))
        x = x + rng.normal(0.0, np.sqrt(n0 / 2.0), size=len(x))
    x = x * (rms / np.sqrt(np.mean(x ** 2)))
    return np.clip(np.round(x * 32767.0), -32768, 32767).astype(np.int16)


def oqpsk_pchannel_pcm(n_frames, fc=8000.0, seed=0, ebn0_db=None, fb=10500.0, Fs=48000.0, phase=0.0, delay=0, return_sus=False):
    bits, sus = pchannel_bits(fb, n_frames, seed, return_sus=True)
    env = oqpsk_envelope(bits, fb, Fs)
    pcm = to_passband_int16(env, fc, Fs, ebn0_db, fb, phase=phase, rng=np.random.default_rng(seed + 12345), delay=delay)
    return (pcm, sus) if return_sus else pcm


def msk_envelope(bits, fb, Fs=48000.0):
    """Complex envelope of the (circular) MSK signal the continuous MSK demodulator decodes to `bits`.
    The demodulator treats MSK as offset QPSK with half-sine pulses (matched filter sin(pi i / (2 SPS)), i < 2 SPS,
    mskdemodulator.cpp:164-170): serial slot n (SPS = Fs/fb samples) carries arm symbol a_n, even slots on the quadrature arm,
    odd slots on the in-phase arm, each pulse two slots long. It emits DiffDecode(imag), then -DiffDecode(real)
    (mskdemodulator.cpp:451-469, DSP.cpp:531-563), i.e. bit_n = NOT([sign a_n != sign a_(n-1)] XOR (n odd)). The pre-coder below
    inverts that; it closes on itself when the number of bits is even and their parity is even."""
    n_bits = len(bits)
    sps = int(round(Fs / fb))
    assert abs(sps - Fs / fb) < 1e-9 and n_bits % 2 == 0
    # sign changes between consecutive arm symbols. The polarity (the final ^ 1) was fixed empirically against the reference
    # demodulator, as SURVEY.md App. D prescribes: the continuous-mode unique-word detector is not polarity invariant
    # (PreambleDetector, aerol.cpp:744-750), so only this variant reaches CRC-valid signal units.
    x = bits.astype(np.int64) ^ (np.arange(n_bits) & 1) ^ 1
    assert (int(x.sum()) & 1) == 0, "bit sequence must have even parity to loop"
    sgn = np.cumsum(x) & 1                                       # sgn_n = sgn_(n-1) ^ x_n with sgn_(-1) = 0
    a = 1.0 - 2.0 * sgn                                          # 0 -> +1
    pulse = np.sin(np.pi * np.arange(2 * sps) / (2.0 * sps))
    L = n_bits * sps
    q = np.zeros(L); i = np.zeros(L)
    for n in range(n_bits):
        idx = (n * sps + np.arange(2 * sps)) % L
        if n & 1:
            i[idx] += a[n] * pulse
        else:
            q[idx] += a[n] * pulse
    return i + 1j * q


def msk_pchannel_pcm(n_frames, fc=2000.0, seed=0, ebn0_db=None, fb=1200.0, Fs=48000.0, phase=0.0, delay=0, return_sus=False):
    """BASELINE cfg 2 signal: differentially pre-coded 600 / 1200 bps MSK P-channel frames, real passband int16."""
    bits, sus = pchannel_bits(fb, n_frames, seed, return_sus=True, loop=True, even_parity=True)
    env = msk_envelope(bits, fb, Fs)
    pcm = to_passband_int16(env, fc, Fs, ebn0_db, fb, phase=phase, rng=np.random.default_rng(seed + 12345), delay=delay)
    return (pcm, sus) if return_sus else pcm


def offset_replicas(pcm, offsets_hz, Fs=48000.0):
    """BASELINE cfg 4 / cfg 5 replicas of a real recording: replica r = Re{ hilbert(x) e^(j 2 pi df_r n / Fs) }, re-quantised to
    int16 (SURVEY.md section 8(d)): a frequency offset applied to the REAL signal. numpy version (tests feed the same arrays to
    the GPU path and to the oracle); bench.py builds the same thing with torch on the device."""
    x = np.asarray(pcm, dtype=np.float64)
    n = len(x)
    X = np.fft.fft(x)
    h = np.zeros(n)
    h[0] = 1.0
    if n % 2 == 0:
        h[n // 2] = 1.0; h[1:n // 2] = 2.0
    else:
        h[1:(n + 1) // 2] = 2.0
    an = np.fft.ifft(X * h)
    t = np.arange(n) / Fs
    out = np.empty((len(offsets_hz), n), dtype=np.int16)
    for r, df in enumerate(offsets_hz):
        y = np.real(an * np.exp(2j * np.pi * float(df) * t))
        out[r] = np.clip(np.round(y), -32768, 32767).astype(np.int16)
    return out


def replica_offsets(r0, r1, span_hz=300.0, seed0=0xB0057):
    """df_r = U(-span, span) from seed seed0 + r (cfg 4: span 300 Hz)."""
    return np.array([np.random.default_rng(seed0 + r).uniform(-span_hz, span_hz) for r in range(r0, r1)])


def wideband_iq(envelopes, offsets_hz, input_rate, env_rate=48000.0, amplitudes=None, ebn0_db=None, fb=10500.0, seed=0,
                iq_format="cs16", noise_ref=0):
    """Complex baseband IQ at input_rate carrying each circular envelope (oqpsk_envelope / msk_envelope, unit power, at
    env_rate) at its offset, plus complex AWGN, quantised as an SDR delivers it: [n, 2] int16 (cs16) or uint8 (cu8, the
    rtl_sdr format, x = ((u - 127.5) + j(v - 127.5)) * 256). Amplitudes (RMS, in cs16 LSB) default to 1000.
    Any input_rate >= env_rate works for which n = len(envelope) * input_rate / env_rate is an integer (2.048 MHz from
    48 kHz, for example). Each envelope is interpolated by zero-padding its FFT to n, so the result still loops seamlessly when every offset is a
    multiple of env_rate / len(envelope). Noise: per-component variance N0 * input_rate / 2 with
    N0 = P / fb / 10^(ebn0_db / 10) of carrier `noise_ref` (P = its amplitude squared, fb its bit rate)."""
    L = len(envelopes[0])
    assert all(len(e) == L for e in envelopes)
    nf = L * float(input_rate) / float(env_rate)
    n = int(round(nf))
    assert abs(nf - n) < 1e-9 * nf and n >= L, "len(envelope) * input_rate / env_rate must be an integer >= len(envelope)"
    amps = np.full(len(envelopes), 1000.0) if amplitudes is None else np.asarray(amplitudes, dtype=np.float64)
    fbs = np.broadcast_to(np.asarray(fb, dtype=np.float64), (len(envelopes),))
    t = np.arange(n, dtype=np.float64)
    x = np.zeros(n, dtype=np.complex128)
    for env, off, a in zip(envelopes, offsets_hz, amps):
        E = np.fft.fft(np.asarray(env, dtype=np.complex128))
        Z = np.zeros(n, dtype=np.complex128)
        h = L // 2
        Z[:h] = E[:h]
        Z[n - (L - h):] = E[h:]
        if L % 2 == 0:                                            # split the Nyquist bin so the result stays band-limited
            Z[h] = 0.5 * E[h]; Z[n - h] = 0.5 * E[h]
        y = np.fft.ifft(Z) * (n / L)                              # n / L = input_rate / env_rate, exact for an integer ratio
        x += a * y * np.exp(2j * np.pi * float(off) * t / float(input_rate))
    if ebn0_db is not None:
        rng = np.random.default_rng(seed)
        n0 = amps[noise_ref] ** 2 / fbs[noise_ref] / (10.0 ** (ebn0_db / 10.0))
        sd = np.sqrt(n0 * float(input_rate) / 2.0)
        x += rng.normal(0.0, sd, n) + 1j * rng.normal(0.0, sd, n)
    out = np.stack([x.real, x.imag], axis=1)
    if iq_format == "cs16":
        return np.clip(np.rint(out), -32768, 32767).astype(np.int16)
    if iq_format == "cu8":
        return np.clip(np.rint(out / 256.0 + 127.5), 0, 255).astype(np.uint8)
    raise ValueError("iq_format must be cs16 or cu8")
