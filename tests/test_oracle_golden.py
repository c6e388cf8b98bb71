"""CPU tests: pin the oracle against everything the reference's own tests hold for this path
(JAERO/tests/fftwrapper_tests.cpp, fftrwrapper_tests.cpp, jfastfir_tests.cpp), against the verbatim
reference build (oracle/_ref) and against committed golden outputs generated from it. What the reference build returns
for these inputs is stored under tests/golden (ref_pins.json through tests/ref_pins.py, jfastfir_golden.npz), so the
comparisons run without the reference."""
import hashlib
import os

import numpy as np
import pytest

from conftest import ROOT, load_excerpt
from oracle import ref, restated
from ref_pins import digest, pinned, same

# JAERO/tests/fftwrapper_tests.cpp:27-29 (captured from JAERO v1.0.4.11)
FFT_IN = [(-0.997497, 0.127171), (-0.613392, 0.617481), (0.170019, -0.040254), (-0.299417, 0.791925), (0.645680, 0.493210), (-0.651784, 0.717887), (0.421003, 0.027070), (-0.392010, -0.970031), (-0.817194, -0.271096), (-0.705374, -0.668203), (0.977050, -0.108615), (-0.761834, -0.990661), (-0.982177, -0.244240), (0.063326, 0.142369), (0.203528, 0.214331), (-0.667531, 0.326090)]
FFT_FWD = [(-4.407605, 0.164434), (2.204298, 2.308064), (-2.713014, -1.356784), (-2.347572, 1.698848), (-2.270577, -0.201056), (1.611736, -2.136282), (-0.902078, 1.606222), (0.335445, -0.964384), (3.648427, 0.230720), (-2.707027, -3.571981), (-1.023916, -0.474082), (1.792787, 2.825653), (-5.574999, 0.226081), (1.119577, -1.518164), (-1.273769, -1.346937), (-3.451670, 4.544378)]
FFT_FWD_BACK = [(-15.959960, 2.034730), (-9.814264, 9.879696), (2.720298, -0.644063), (-4.790674, 12.670797), (10.330882, 7.891354), (-10.428541, 11.486190), (6.736045, 0.433119), (-6.272164, -15.520493), (-13.075106, -4.337535), (-11.285989, -10.691244), (15.632801, -1.737846), (-12.189337, -15.850581), (-15.714835, -3.907834), (1.013215, 2.277902), (3.256447, 3.429304), (-10.680502, 5.217444)]
TOL = 0.00001   # doubles_equal_threshold in the reference tests


def _fft(lib_fn, x, inverse):
    a = np.ascontiguousarray(np.asarray(x, dtype=np.float64))
    o = np.zeros_like(a)
    lib_fn(len(a), int(inverse), a.ctypes.data, o.ctypes.data)
    return o


def test_fft_known_answer_restated():
    """Test_FFTWrapper (fftwrapper_tests.cpp:23-54) against the oracle's FFT: forward e^-j, inverse unnormalised."""
    L = restated.lib()
    fwd = _fft(L.jor_fft, FFT_IN, False)
    assert np.abs(fwd - np.asarray(FFT_FWD)).max() < TOL
    back = _fft(L.jor_fft, fwd, True)
    assert np.abs(back - np.asarray(FFT_FWD_BACK)).max() < TOL


def test_fft_known_answer_reference_wrapper():
    """Same vector through the reference's own FFTWrapper over the restated JFFT; the oracle's FFT gives the same values."""
    def run():
        fwd = _fft(ref.lib().jref_fft, FFT_IN, False)
        return [fwd, _fft(ref.lib().jref_fft, fwd, True)]
    fwd, back = (np.asarray(v) for v in pinned("oracle/fft_wrapper", run))
    assert np.abs(fwd - np.asarray(FFT_FWD)).max() < TOL
    assert np.abs(back - np.asarray(FFT_FWD_BACK)).max() < TOL
    L = restated.lib()
    assert np.abs(_fft(L.jor_fft, FFT_IN, False) - fwd).max() < 1e-12
    assert np.abs(_fft(L.jor_fft, fwd, True) - back).max() < 1e-12


def test_fftr_wrapper_semantics():
    """Test_FFTrWrapper (fftrwrapper_tests.cpp:24-55): r2c zeroes bins above N/2, c2r scales by N."""
    x = np.array([v[0] for v in FFT_IN])

    def run():
        L = ref.lib()
        out = np.zeros((16, 2))
        L.jref_fftr_forward(16, x.ctypes.data, out.ctypes.data)
        back = np.zeros(16)
        L.jref_fftr_inverse(16, out.ctypes.data, back.ctypes.data)
        return [out.ravel(), back]
    out, back = (np.asarray(v) for v in pinned("oracle/fftr_wrapper", run))
    out = out.reshape(16, 2)
    full = np.fft.fft(x)
    assert np.abs((out[:9, 0] + 1j * out[:9, 1]) - full[:9]).max() < TOL
    assert np.all(out[9:] == 0)
    assert np.abs(back - 16 * x).max() < TOL


def test_jfastfir_golden():
    """Test_JFastFir (jfastfir_tests.cpp:31-58): 10 000-sample golden from JAERO v1.0.4.11 (the reference's own data files,
    printed to 6 significant digits; stored as float32 in tests/golden/jfastfir_golden.npz, every 5th expected output) through
    the restated JFastFir with the restated root-raised-cosine kernel. The reference only checks n >= 4096; the restated
    JFastFir matches everywhere."""
    z = np.load(os.path.join(ROOT, "tests", "golden", "jfastfir_golden.npz"))
    six = lambda a: np.array([float("%.6g" % v) for v in a.ravel()]).reshape(a.shape)    # the data files' decimal values
    gi, go, step = six(z["input"]), six(z["expected_output"]), int(z["step"])
    Fs, fb = float(z["Fs"]), float(z["fb"])
    buf = np.ascontiguousarray(gi)
    restated.lib().jor_jfastfir_rrc(0.6, 2048, Fs, fb / 2, 4096, buf.ctypes.data, len(buf))
    got = buf[::step]
    assert np.abs(got[4096 // step:] - go[4096 // step:]).max() < TOL
    assert np.abs(got[:4096 // step] - go[:4096 // step]).max() < TOL


def test_dsp_primitive_semantics():
    """SURVEY.md P4: FIR one-sample extra delay, qRound, RRC taps and trig tables identical in oracle and reference."""
    R = restated.lib()
    taps = np.array([1.0, 2.0, 3.0, 4.0]); x = np.array([1.0, 0, 0, 0, 0, 0])

    def fir():
        y = np.zeros(6)
        ref.lib().jref_fir(taps.ctypes.data, 4, x.ctypes.data, y.ctypes.data, 6)
        return y
    assert pinned("oracle/fir_impulse", fir) == [0, 4, 3, 2, 1, 0]
    vals = (-0.5, 0.5, 1.5, -1.5, 127.49, 254.5, -3.2)
    q = pinned("oracle/qround", lambda: [ref.lib().jref_qround(v) for v in vals])
    assert q == [R.jor_qround(v) for v in vals]
    assert q[0] == 0 and q[1] == 1                                    # qRound(-0.5), qRound(0.5)

    def rrc():
        a = np.zeros(64)
        return [ref.lib().jref_rrc_design(1.0, 55, 48000.0, 5250.0, a.ctypes.data, 64), a]
    b = np.zeros(64)
    nb = R.jor_rrc_design(1.0, 55, 48000.0, 5250.0, b.ctypes.data, 64)
    assert nb == 55 and same([nb, b], "oracle/rrc_taps", rrc)

    def trig():
        s1 = np.zeros(19999); c1 = np.zeros(19999)
        ref.lib().jref_trig_tables(s1.ctypes.data, c1.ctypes.data)
        return [s1, c1]
    s2 = np.zeros(19999); c2 = np.zeros(19999)
    R.jor_trig_tables(s2.ctypes.data, c2.ctypes.data)
    assert same([s2, c2], "oracle/trig_tables", trig)


def _run_restated(case, pcm):
    if case["kind"].startswith("burst"):
        d = restated.OracleDemod(case["kind"], **case["kw"])
        for a in range(0, len(pcm), case["chunk"]):
            d.write(pcm[a:a + case["chunk"]])
        return d.take_soft(), d.state(), np.zeros(0)
    d = restated.OracleDemod(case["kind"], **case["kw"])
    sched = {int(a): int(v) for a, v in case["dcd_schedule"]}
    for a in range(0, len(pcm), case["chunk"]):
        if a in sched:
            d.set_dcd(sched[a])
        d.write(pcm[a:a + case["chunk"]])
    return d.take_soft(), d.state(), d.take_cfe_log()


@pytest.mark.parametrize("name", ["oqpsk_10500", "oqpsk_10500_noafc_dcd", "oqpsk_8400", "msk_600", "msk_1200", "msk_1200_noafc_dcd",
                                  "burst_msk_1200_a", "burst_msk_1200_b", "burst_oqpsk_10500"])
def test_restated_oracle_matches_reference_golden(golden, name):
    """The restatement reproduces the verbatim reference bit for bit on the recordings (soft bits, coarse
    estimates, loop state) — golden values were produced by oracle/_ref (tools/make_golden_outputs.py)."""
    case = golden[name]
    soft, state, cfe = _run_restated(case, load_excerpt(case["excerpt"]))
    assert len(soft) == case["n_soft"]
    assert hashlib.sha256(soft.astype("<i2").tobytes()).hexdigest() == case["soft_sha256"]
    if not case["kind"].startswith("burst"):
        assert hashlib.sha256(np.asarray(cfe, dtype="<f8").tobytes()).hexdigest() == case["cfe_log_sha256"]
    else:
        assert int((soft < 0).sum()) >= 2                      # burst start markers (-1) survive
    for k, v in case["state"].items():
        assert state[k] == v, k


@pytest.mark.parametrize("name", ["oqpsk_10500", "msk_600", "msk_1200"])
def test_restated_oracle_matches_reference_live(golden, name):
    """Same comparison on the first 6 s without a DCD schedule, against the reference library run on it (in a fresh
    process: the reference has function statics) and stored in tests/golden/ref_pins.json."""
    import multiprocessing as mp
    case = golden[name]
    pcm = load_excerpt(case["excerpt"])[:48000 * 6]

    def run():
        with mp.get_context("spawn").Pool(1) as pool:
            rs, rstate, rcfe = pool.apply(ref.run_demod_job, ((case["kind"], case["kw"], pcm, case["chunk"], None),))
        return [rs, rcfe, rstate]
    soft, state, cfe = _run_restated(dict(case, dcd_schedule=[]), pcm)
    rs, rcfe, rstate = pinned("oracle/demod_6s_" + name, run)
    assert digest(soft) == rs and digest(cfe) == rcfe
    for k in rstate:
        assert rstate[k] == state[k], k


@pytest.mark.parametrize("name", ["oqpsk_10500", "msk_600"])
def test_pchannel_decode_yields_crc_valid_signal_units(golden, name):
    """Pins the restated libcorrect (parity unpinned upstream): the reference's own recordings decode to
    CRC-16-valid 12-byte SUs in every frame after lock, identical to the committed golden."""
    case = golden[name]
    soft, _, _ = _run_restated(case, load_excerpt(case["excerpt"]))
    p = restated.OraclePChannel(case["kw"]["fb"])
    p.process(soft)
    su, ok, fr = p.take_sus()
    assert len(ok) == case["n_su"] and int(ok.sum()) == case["n_su_crc_ok"]
    assert hashlib.sha256(su.tobytes() + ok.astype("<i4").tobytes()).hexdigest() == case["su_sha256"]
    per_frame = {f: ok[fr == f] for f in np.unique(fr)}
    good_frames = [f for f, v in per_frame.items() if v.all()]
    assert len(good_frames) >= len(per_frame) - 4          # only the first frames after lock may fail
    assert all(per_frame[f].all() for f in sorted(per_frame)[4:])


def test_viterbi_restated_equals_reference_wrapper():
    """Restated Decode_Continuous == the reference's JConvolutionalCodec (verbatim) over the same libcorrect: one decoder
    object over consecutive blocks, so the state carried between calls is compared too."""
    rng = np.random.default_rng(3)
    blocks = [rng.integers(0, 256, size=n, dtype=np.uint8) for n in (4992, 4992, 576, 384, 4992)]

    def run():
        a = ref.RefCodec(24)
        return [a.decode_continuous(soft) for soft in blocks]
    b = restated.OracleViterbi(24)
    assert same([b.decode_continuous(soft) for soft in blocks], "oracle/viterbi_continuous", run)


def test_viterbi_roundtrip_and_error_correction():
    rng = np.random.default_rng(5)
    msg = rng.integers(0, 256, size=300, dtype=np.uint8)
    enc = restated.conv_encode(msg)
    soft = (enc * 255).astype(np.uint8)
    dec = restated.conv_decode_soft(soft)
    assert np.array_equal(dec[:2400], np.unpackbits(msg))
    noisy = np.clip(np.round((enc * 2.0 - 1) * 70 + 128 + rng.normal(0, 40, size=len(enc))), 0, 255).astype(np.uint8)
    dec = restated.conv_decode_soft(noisy)
    assert np.array_equal(dec[:2400], np.unpackbits(msg))


def test_synthetic_pchannel_signal_decodes():
    """The transmit chain (jaero_b200/synth.py) inverts AeroL::Decode: the oracle recovers the transmitted SUs."""
    from jaero_b200 import synth
    pcm, sus = synth.oqpsk_pchannel_pcm(10, fc=8000.0, seed=11, ebn0_db=10.0, return_sus=True)
    d = restated.OracleDemod("oqpsk", fb=10500, freq_center=8000, lockingbw=10500, fft_power=14, signalthreshold=0.65)
    for a in range(0, len(pcm), 4800):
        d.write(pcm[a:a + 4800])
    p = restated.OraclePChannel(10500)
    p.process(d.take_soft())
    b, ok, _ = p.take_sus()
    tx = {bytes(x) for x in sus.reshape(-1, 12)}
    assert ok.sum() >= 26 * 3
    assert all(bytes(x) in tx for x in b[ok == 1])
    assert abs(d.state()["ebno"] - 10.0) < 1.0


@pytest.mark.parametrize("name", ["burst_msk_1200_a", "burst_msk_1200_b", "burst_oqpsk_10500"])
def test_rt_channel_oracle_decodes_crc_valid_packets(golden, name):
    """SURVEY 8(f)2: the restated burst branch of AeroL::Decode + RTChannelDeleaveFECScram turns the reference's soft bits
    into T packets whose header and signal-unit CRC-16s verify (self-certifying: de-interleaver, Viterbi restatement,
    scrambler and CRC all have to be right), identical to the committed golden, and independent of how the stream is cut."""
    case = golden[name]
    soft, _, _ = _run_restated(case, load_excerpt(case["excerpt"]))
    rt = restated.OracleRTChannel(case["kw"]["fb"])
    rt.process(soft)
    pk = rt.packets()
    assert len(pk) == len(case["rt_packets"]) >= 2
    for q, g in zip(pk, case["rt_packets"]):
        assert q["type"] == g["type"] == 2 and q["nsus"] == g["nsus"] and len(q["bytes"]) == g["n_bytes"]
        assert hashlib.sha256(q["bytes"].tobytes()).hexdigest() == g["sha256"]
    rt2 = restated.OracleRTChannel(case["kw"]["fb"])
    for a in range(0, len(soft), 33):
        rt2.process(soft[a:a + 33], vector_semantics=True)
    pk2 = rt2.packets()
    assert len(pk2) == len(pk) and all(np.array_equal(a["bytes"], b["bytes"]) for a, b in zip(pk, pk2))


def test_c_channel_oracle_decodes_crc_valid_signal_units(golden):
    """SURVEY 8(f)3: restated AeroL::DecodeC on the 8400 bps recording: dual-UW ambiguity detector, 16 x (64 x 4)
    de-interleave, rate-3/4 de-puncturing, continuous Viterbi, delay line, scrambler -> sub-band signal units whose
    CRC-16 verifies (self-certifying), identical to the committed golden."""
    case = golden["oqpsk_8400"]
    soft, _, _ = _run_restated(case, load_excerpt(case["excerpt"]))
    cc = restated.OracleCChannel()
    for a in range(0, len(soft), 1000):
        cc.process(soft[a:a + 1000])
    su, cok, voice = cc.take_frames()
    g = case["c_frames"]
    assert len(su) == g["n_frames"] >= 5 and int(cok.sum()) == g["n_su_crc_ok"] >= 10
    assert hashlib.sha256(su.tobytes() + cok.astype("<i4").tobytes() + voice.tobytes()).hexdigest() == g["sha256"]


@pytest.mark.parametrize("fb", [1200, 10500])
@pytest.mark.parametrize("invert", [False, True])
def test_rt_channel_oracle_known_answer_r_packet(fb, invert):
    """A synthetic R-channel packet (encoder written from the specification side: CRC-16, scrambler, K=7 109/79 code, 64 x 5
    interleaver, unique word) is decoded back to its 19 bytes by the restated receive chain, in either signal polarity."""
    from conftest import synthetic_r_packet_stream
    payload = (np.arange(17) * 37 + 11).astype(np.uint8)
    soft = synthetic_r_packet_stream(fb, payload, invert=invert)
    rt = restated.OracleRTChannel(fb)
    rt.process(soft)
    pk = rt.packets()
    assert len(pk) == 1 and pk[0]["type"] == 1 and len(pk[0]["bytes"]) == 19
    assert np.array_equal(pk[0]["bytes"][:17], payload)


@pytest.mark.parametrize("fb", [1200, 600])
def test_msk_generator_known_answer_through_the_oracle(fb):
    """BASELINE cfg 2 signal model: the differentially pre-coded MSK P-channel generator (jaero_b200.synth) and the oracle's
    continuous MSK demodulator + P-channel layer are inverse to each other: every CRC-valid signal unit that comes out is one
    that went in, in order, and after lock all of them come out (Eb/N0 = 12 dB)."""
    from jaero_b200 import synth
    n_frames = 8
    pcm, sus = synth.msk_pchannel_pcm(n_frames, fc=2011.0, seed=77 + fb, ebn0_db=12.0, fb=float(fb), phase=2.2, delay=5, return_sus=True)
    pcm = np.tile(pcm, 2)                                        # the frame sequence loops seamlessly (tail-biting code, even parity)
    d = restated.OracleDemod("msk", fb=fb, freq_center=2000.0, lockingbw=1800 if fb == 1200 else 900, fft_power=13, signalthreshold=0.5)
    p = restated.OraclePChannel(fb)
    for a in range(0, len(pcm), 4800):
        d.write(pcm[a:a + 4800]); p.process(d.take_soft()); d.set_dcd(p.dcd)
    su, ok, fr = p.take_sus()
    sent = [bytes(x) for x in sus.reshape(-1, 12)] * 2
    got = [bytes(x) for x in su[ok.astype(bool)]]
    assert len(got) >= len(sent) - 4 * sus.shape[1]              # at most the first frames (lock + decoder latency) are missing
    # in order: got is a contiguous run of `sent` (which repeats with the loop)
    k0 = sent.index(got[0])
    assert got == sent[k0:k0 + len(got)]
    assert int(ok.sum()) == len(ok) - int((~ok.astype(bool))[:2 * sus.shape[1]].sum())   # no CRC failure after the first two frames
