"""CPU tests: the restated frame-layer oracle (oracle/restated/fec_oracle.cpp), piece by piece, against the reference's OWN
helper classes compiled verbatim from JAERO/aerol.h:283-895 + aerol.cpp:523-902,2505-2524 (oracle/ref_fec_driver.cpp ->
oracle/_ref/libjaero_ref_fec.so): CRC-16 (bytes and bits), scrambler, interleaver, puncturing, the three unique-word
detectors and the R/T packet decoder RTChannelDeleaveFECScram (trial de-interleave + Viterbi + descramble + CRC at every
candidate length). Random inputs, recorded soft bits and known-answer packets. The reference's results on these inputs are
stored in tests/golden/ref_pins.json (tests/ref_pins.py), so the tests need neither the reference nor oracle/_ref."""
import ctypes
import os

import numpy as np
import pytest

from conftest import ROOT, load_excerpt, synthetic_r_packet_stream
from oracle import restated
from ref_pins import RECORD, pinned, same

SO = os.path.join(ROOT, "oracle", "_ref", "libjaero_ref_fec.so")
UW = 0xE15AE893
C_PRE1, C_PRE2 = 216866263330005, 3012071630031408          # aerol.cpp:953-954


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


@pytest.fixture(scope="module")
def F():
    """the reference build, loaded only to record its results (ref_pins.RECORD)"""
    if not RECORD:
        return None
    L = ctypes.CDLL(SO)
    L.jfec_rt_new.restype = ctypes.c_void_p
    for n in ("jfec_rt_free", "jfec_rt_reset"):
        getattr(L, n).argtypes = [ctypes.c_void_p]
    L.jfec_rt_update.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int]
    L.jfec_rt_info.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]
    L.jfec_detect.argtypes = [ctypes.c_int, ctypes.c_ulonglong, ctypes.c_ulonglong, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
    L.jfec_crc_bytes.restype = ctypes.c_uint
    return L


@pytest.fixture(scope="module")
def R():
    L = restated.lib()
    L.jor_pin_rt_new.restype = ctypes.c_void_p
    for n in ("jor_pin_rt_free", "jor_pin_rt_reset"):
        getattr(L, n).argtypes = [ctypes.c_void_p]
    L.jor_pin_rt_update.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int]
    L.jor_pin_rt_info.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]
    return L


def test_crc16_bytes_and_bits(F, R):
    rng = np.random.default_rng(1)
    blocks = [rng.integers(0, 256, size=n, dtype=np.uint8) for n in (1, 10, 12, 17, 19, 64) for _ in range(50)]
    assert same([R.jor_crc16(_p(b), len(b)) for b in blocks], "fec/crc16_bytes", lambda: [F.jfec_crc_bytes(_p(b), len(b)) for b in blocks])
    from jaero_b200 import synth
    words = []
    for nbits in (8 * 19, 8 * 12, 48 + 96 * 3):
        for k in range(60):
            body = rng.integers(0, 2, size=nbits - 16).astype(np.int32)
            by = np.packbits(body.astype(np.uint8), bitorder="little")
            c = synth.crc16(by) if (nbits - 16) % 8 == 0 else 0
            bits = np.concatenate([body, np.array([(c >> i) & 1 for i in range(16)], dtype=np.int32)]).astype(np.int32)
            if k % 3 == 0:
                bits[rng.integers(0, nbits)] ^= 1
            words.append(bits)
    assert same([R.jor_pin_crc_bits_check(_p(w), len(w)) for w in words], "fec/crc16_bits",
                lambda: [F.jfec_crc_bits_check(_p(w), len(w)) for w in words])
    good = np.concatenate([np.zeros(136, dtype=np.int32), np.array([(synth.crc16(np.zeros(17, dtype=np.uint8)) >> i) & 1 for i in range(16)], dtype=np.int32)])
    assert pinned("fec/crc16_bits_good", lambda: F.jfec_crc_bits_check(_p(good), 152)) == 1 == R.jor_pin_crc_bits_check(_p(good), 152)


def test_scrambler_sequence_and_piecewise_update(F, R):
    seq = np.zeros(5000, dtype=np.int32)
    R.jor_pin_scrambler(_p(seq), 5000)
    sizes = np.array([288, 288, 1, 999, 2496, 928], dtype=np.int32)
    def ref():
        bits = np.zeros(int(sizes.sum()), dtype=np.int32)             # scrambling zeros returns the sequence itself
        F.jfec_scramble(_p(bits), _p(sizes), len(sizes))
        return bits
    assert same(seq, "fec/scrambler", ref)
    from jaero_b200 import synth
    assert np.array_equal(synth.scrambler_sequence(5000), seq.astype(np.uint8))


@pytest.mark.parametrize("cols", [6, 9, 78, 5, 3, 4])
def test_deinterleaver_matches_reference(F, R, cols):
    rng = np.random.default_rng(cols)
    for setsize in (cols, 95):
        block = rng.integers(0, 256, size=64 * cols).astype(np.int32)
        if setsize != cols:
            block = np.concatenate([block, rng.integers(0, 256, size=64 * (setsize - cols)).astype(np.int32)])
        def ref():
            out = np.zeros(64 * setsize, dtype=np.uint8)
            n = F.jfec_deinterleave_ba(_p(block), len(block), setsize, cols, _p(out))
            return [n >= 64 * cols, out[:64 * cols]]
        got = np.zeros(64 * cols, dtype=np.uint8)
        R.jor_deinterleave(_p(np.ascontiguousarray(block[:64 * cols])), cols, _p(got))
        assert same([True, got], "fec/deinterleave_%d_%d" % (cols, setsize), ref)
    # and the generator's interleaver is the reference's
    from jaero_b200 import synth
    x = rng.integers(0, 2, size=64 * cols).astype(np.int32)

    def ref_il():
        o = np.zeros(64 * cols, dtype=np.int32)
        return [F.jfec_interleave(_p(x), len(x), cols, _p(o)), o]
    assert same([64 * cols, synth.interleave(x.astype(np.uint8), cols)], "fec/interleave_%d" % cols, ref_il)


def test_c_channel_block_deinterleave_and_depuncture(F, R):
    """DecodeC: 16 blocks of 4 x 64 -> deinterleave_ba(block, 4) each, appended, then depunture_soft_block(.., 4) (aerol.cpp:2306-2327)"""
    rng = np.random.default_rng(5)
    frame = rng.integers(0, 256, size=4096).astype(np.int32)
    got = np.zeros(6000, dtype=np.uint8)
    ng = R.jor_pin_c_code_order(_p(frame), _p(got))
    def ref():
        dele = []
        for b in range(16):
            o = np.zeros(64 * 95, dtype=np.uint8)
            n = F.jfec_deinterleave_ba(_p(np.ascontiguousarray(frame[256 * b:256 * b + 256])), 256, 4, 4, _p(o))
            dele.append(o[:256].copy()); assert n == 256
        src = np.concatenate(dele); sizes = np.array([len(src)], dtype=np.int32)
        out = np.zeros(6000, dtype=np.uint8)
        nr = F.jfec_depuncture(_p(src), _p(sizes), 1, 4, _p(out))
        return [nr, out[:nr]]
    assert same([ng, got[:ng]], "fec/c_code_order", ref)


@pytest.mark.parametrize("kind,tol", [(0, 0), (1, 0), (3, 4), (2, 6)])
def test_unique_word_detectors_on_random_and_recorded_bits(F, R, kind, tol):
    """kind 0 PreambleDetector, 1 PreambleDetectorPhaseInvariant (tol 0: continuous P-channel 10.5k), 3 the same with tolerance 4
    (burst R/T), 2 OQPSKPreambleDetectorAndAmbiguityCorrection (C-channel). Hits, polarity flags and the state after hits."""
    rng = np.random.default_rng(10 + kind)
    uw = np.array([(UW >> (31 - i)) & 1 for i in range(32)], dtype=np.int32)
    w1 = np.array([(C_PRE1 >> (51 - i)) & 1 for i in range(52)], dtype=np.int32)
    w2 = np.array([(C_PRE2 >> (51 - i)) & 1 for i in range(52)], dtype=np.int32)
    pieces = [rng.integers(0, 2, size=700).astype(np.int32)]
    for k in range(12):
        word = (uw if kind != 2 else (w1 if k % 2 else w2)).copy()
        if k % 3 == 1:
            word = 1 - word                                          # inverted
        nerr = [0, 1, tol, tol + 1][k % 4]
        if nerr:
            word[rng.choice(len(word), size=nerr, replace=False)] ^= 1
        pieces += [word, rng.integers(0, 2, size=int(rng.integers(1, 300))).astype(np.int32)]
    soft = load_excerpt("burst_msk_1200_a")[:20000]
    pieces.append((soft > 0).astype(np.int32))
    bits = np.ascontiguousarray(np.concatenate(pieces))
    n = len(bits)
    ref_kind = {0: 0, 1: 1, 3: 1, 2: 2}[kind]

    def ref():
        o1 = np.zeros(n, dtype=np.int32); i1 = np.zeros(n, dtype=np.int32)
        F.jfec_detect(ref_kind, UW if kind != 2 else C_PRE1, C_PRE2, 32 if kind != 2 else 52, tol, _p(bits), n, _p(o1), _p(i1))
        return [o1, int(o1.sum()), i1 if kind else []]
    o2 = np.zeros(n, dtype=np.int32); i2 = np.zeros(n, dtype=np.int32)
    R.jor_pin_detect(kind, tol, _p(bits), n, _p(o2), _p(i2))
    assert same([o2, int(o2.sum()), i2 if kind else []], "fec/detect_%d_%d" % (kind, tol), ref) and o2.sum() >= 3


def _rt_run(L, new, reset, update, info, free, fb, soft, msk):
    h = new() if fb is None else new(fb)
    res = []
    reset(h)
    buf = np.zeros(512, dtype=np.uint8); nsus = ctypes.c_int(0)
    for v in soft:
        r = update(h, msk, int(v))
        if r != 8:                                                   # not `Nothing`
            n = info(h, _p(buf), 512, ctypes.byref(nsus))
            res.append((len(res), r, n, nsus.value if r == 5 else -1, bytes(buf[:min(n, 512)])))   # numberofsus is only set for T packets (uninitialised otherwise in the reference)
            if r & 1:
                reset(h)
    free(h)
    return res


def _rt_key(res):
    """what the two decoders must agree on: every report's position, result code, length and number of SUs, and the payload
    bytes of every packet"""
    return [list(x[:4]) + [x[4] if x[1] & 1 else b""] for x in res]


@pytest.mark.parametrize("fb", [1200, 10500])
def test_rt_packet_decoder_matches_reference_class(F, R, fb):
    """RTChannelDeleaveFECScram::update / updateMSK (aerol.h:631-877) against RTChannelOracle::rt_update / rt_updateMSK: the result
    code after every soft bit, and infofield / numberofsus whenever something is reported; known-answer R packets, random soft
    bits (every trial fails) and noisy packets."""
    msk = 0 if fb == 10500 else 1
    rng = np.random.default_rng(fb)
    streams = []
    for k in range(3):
        s = synthetic_r_packet_stream(fb, ((np.arange(17) * (3 + k) + k) % 256).astype(np.uint8), invert=False)
        uwlen = 64 if fb == 10500 else 32
        body = s[1 + 80 + uwlen:]                                    # marker, filler, unique word stripped: the block starts here
        if k == 2:
            body = np.clip(body + rng.normal(0, 40, size=len(body)), 0, 255).astype(np.int16)
        streams.append(body.astype(np.int32))
    streams.append(rng.integers(0, 256, size=64 * 12).astype(np.int32))
    for k, soft in enumerate(streams):
        a = lambda: _rt_key(_rt_run(F, F.jfec_rt_new, F.jfec_rt_reset, F.jfec_rt_update, F.jfec_rt_info, F.jfec_rt_free, None, soft, msk))
        b = _rt_run(R, R.jor_pin_rt_new, R.jor_pin_rt_reset, R.jor_pin_rt_update, R.jor_pin_rt_info, R.jor_pin_rt_free, fb, soft, msk)
        assert same(_rt_key(b), "fec/rt_decoder_%d_%d" % (fb, k), a)


def test_rt_t_packets_from_the_burst_recording(F, R):
    """Soft bits the reference's burst demodulator emits on samples/1200bps_burst_sample1.wav: cut at the start-of-burst markers,
    un-inverted per burst by the unique word, fed to both packet decoders bit by bit."""
    case_kw = dict(fb=1200.0, freq_center=1000.0, lockingbw=1800.0, signalthreshold=0.6)
    soft, _, _ = restated.run_demod_job(("burst_msk", case_kw, load_excerpt("burst_msk_1200_a"), 48000))
    marks = list(np.nonzero(soft < 0)[0]) + [len(soft)]
    tried = 0
    for k in range(len(marks) - 1):
        seg = soft[marks[k] + 1:marks[k + 1]].astype(np.int32)
        hard = (seg >= 128).astype(np.int64)
        uw = np.array([(UW >> (31 - i)) & 1 for i in range(32)])
        pos = None
        for i in range(0, min(len(hard) - 32, 400)):
            d = int((hard[i:i + 32] ^ uw).sum())
            if d <= 4 or d >= 28:
                pos, inv = i + 32, d >= 28
                break
        if pos is None:
            continue
        body = seg[pos:]
        if inv:
            body = np.where(body == 128, 128, 255 - body)
        a = lambda: _rt_key(_rt_run(F, F.jfec_rt_new, F.jfec_rt_reset, F.jfec_rt_update, F.jfec_rt_info, F.jfec_rt_free, None, body, 1))
        b = _rt_run(R, R.jor_pin_rt_new, R.jor_pin_rt_reset, R.jor_pin_rt_update, R.jor_pin_rt_info, R.jor_pin_rt_free, 1200, body, 1)
        assert same(_rt_key(b), "fec/rt_recording_%d" % k, a)
        tried += 1
    assert tried >= 2
