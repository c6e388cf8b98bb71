"""Device channelizer at rational rates (output_rate / input_rate = L/M) on the GPU: against the float64 polyphase
definition (tests/chan_poly_ref.py), independence from how the input is cut into writes and from where a channel sits in
the tile, selectivity, and rtl_sdr-rate cu8 IQ through channelizer -> demodulator -> P-channel layer to CRC-valid signal units."""
import numpy as np
import pytest

from chan_poly_ref import chan_poly_ref, n_outputs
from chan_ref import iq_to_complex
from conftest import has_cuda
from test_channelizer_gpu import _amp, _decode_oracle, _dev, _noise_and_carriers, _offsets, _pchan_sus

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not has_cuda(), reason="needs a CUDA device")]


def _jb():
    import jaero_b200
    return jaero_b200


CASES = [  # iq_format, input_rate, output_rate, audio_hz, passband_hz
    ("cs16", 2.048e6, 48000.0, 12000.0, 12000.0),
    ("cu8", 2.048e6, 48000.0, 12000.0, 12000.0),
    ("cu8", 1.024e6, 48000.0, 12000.0, 3000.0),
    ("cs16", 2.5e6, 48000.0, 12000.0, 12000.0),
    ("cu8", 3e6, 48000.0, 12000.0, 10000.0),
    ("cs16", 3e6, 24000.0, 6000.0, 3000.0),             # 3 MHz is 125 x 24 kHz: L = 1 through the same path
]


@pytest.mark.parametrize("case", CASES, ids=["%s-%g-%d-%d" % (c[0], c[1], c[2], c[4]) for c in CASES])
def test_rational_channelizer_matches_definition(case):
    jb = _jb()
    fmt, fs, fo, audio, pb = case
    L, M = jb.channelizer_ratio(fs, output_rate=fo, audio_hz=audio, passband_hz=pb)
    rng = np.random.default_rng(L * 1000 + M)
    C = 70
    off = _offsets(rng, C, fs, pb)
    n = 700 * M // L + 13
    iq = _noise_and_carriers(rng, n, fs, fmt)
    ch = jb.Channelizer(off, fs, output_rate=fo, audio_hz=audio, passband_hz=pb, iq_format=fmt, gain=0.8)
    assert ch.ratio == (L, M) and ch.D == (M if L == 1 else None)
    ch.write(iq)
    got = ch.read()
    h = jb.channelizer_taps(fs, output_rate=fo, audio_hz=audio, passband_hz=pb)
    want = chan_poly_ref(iq_to_complex(iq, fmt), h, L, M, off, fs, output_rate=fo, audio_hz=audio, gain=0.8)
    assert got.shape == want.shape == (C, n_outputs(n, L, M))
    d = np.abs(got.astype(np.int32) - want)
    assert d.max() <= 1, np.unravel_index(np.argmax(d), d.shape)
    assert np.mean(d == 0) >= 0.99, np.mean(d == 0)
    assert np.abs(want).max() > 1000                      # the comparison covers large values, not only noise
    ch.close()


@pytest.mark.parametrize("fs", [2.048e6, 2.5e6])
def test_rational_chunking_and_device_feed_are_bit_identical(fs):
    jb = _jb()
    L, M = jb.channelizer_ratio(fs)
    rng = np.random.default_rng(L)
    off = _offsets(rng, 70, fs, 12000.0)
    n = 40 * M + 29
    iq = _noise_and_carriers(rng, n, fs, "cs16")
    one = jb.Channelizer(off, fs)
    one.write(iq)
    ref = one.read()
    sizes = [1, 2, M - 1, M, M + 1, 4097, M // L + 5]
    cuts = np.cumsum(sizes)
    ends = [n_outputs(int(e), L, M) for e in cuts]
    assert any(e % L for e in ends)                        # some write ends part-way through the L residue classes
    pieces = np.split(iq, cuts)
    many = jb.Channelizer(off, fs)
    dev = jb.Channelizer(off, fs)
    d_iq = _dev(iq)
    got, got_dev = [], []
    pos = 0
    for p in pieces:
        many.write(p)
        got.append(many.read())
        dev.write_device(d_iq.data_ptr() + pos * 4, len(p))
        got_dev.append(dev.read())
        pos += len(p)
    assert any(g.shape[1] == 0 for g in got)               # some writes end without an output
    got, got_dev = np.concatenate(got, axis=1), np.concatenate(got_dev, axis=1)
    assert np.array_equal(got, ref)
    assert np.array_equal(got_dev, ref)
    assert many.launches <= 2 * len(pieces) and dev.launches <= 2 * len(pieces)
    for c in (one, many, dev):
        c.close()


def test_rational_rows_do_not_depend_on_position():
    jb = _jb()
    fs = 2.048e6
    L, M = jb.channelizer_ratio(fs)
    base = np.array([-701234.25, -3000.5, 17.0, 650001.75])
    off = np.tile(base, 256)                               # 1024 channels, 4 interleaved offsets
    rng = np.random.default_rng(12)
    iq = _noise_and_carriers(rng, 400 * M // L + 5, fs, "cs16")
    ch = jb.Channelizer(off, fs)
    ch.write(iq)
    out = ch.read()
    for c in range(4):
        assert np.array_equal(out[c::4], np.broadcast_to(out[c], out[c::4].shape)), c
    ch.close()


def test_rational_selectivity_with_tones():
    jb = _jb()
    fs, pb, audio = 2.048e6, 12000.0, 12000.0
    L, M = jb.channelizer_ratio(fs)
    fp = pb / 2
    f_s = min(2 * audio, 48000.0 - 2 * audio) - fp
    centre = 123456.0
    A, gain = 20000.0, 1.5
    deltas = [0.99 * fp, -0.99 * fp, f_s, -f_s, 1.5 * f_s, -3 * f_s, 100000.0, -400000.0]
    n = 4000 * M // L
    t = np.arange(n)
    rows = []
    for dlt in deltas:                                     # one tone at a time
        x = A * np.exp(2j * np.pi * (centre + dlt) * t / fs)
        iq = np.clip(np.rint(np.stack([x.real, x.imag], axis=1)), -32768, 32767).astype(np.int16)
        c1 = jb.Channelizer([centre], fs, passband_hz=pb, gain=gain)
        c1.write(iq)
        rows.append(c1.read()[0, 100:])                   # past the filter's start-up (Tp = 620 inputs < 100 outputs)
        c1.close()
    full = gain * A
    for dlt, r in zip(deltas[:2], rows[:2]):
        db = 20 * np.log10(_amp(r) / full)
        assert abs(db) <= 0.05, (dlt, db)
    for dlt, r in zip(deltas[2:], rows[2:]):
        a = _amp(r)
        assert 20 * np.log10(max(a, 1e-9) / full) <= -58.0, (dlt, a)
    assert _amp(rows[2]) > 10.0                            # the suppressed tone is still tens of LSB, not rounded away


def test_rtl_sdr_rate_cu8_iq_to_signal_units():
    """2.048 MHz cu8 (the rtl_sdr default), 6 s (two loops of 3 s): 13 OQPSK 10.5k carriers (one of them 30 dB stronger,
    25 kHz from a weak one) and 4 MSK 1200 carriers at Eb/N0 10 dB, two handles on the same device IQ, each with its own
    stream, batch and P-channel layer."""
    jb = _jb()
    import torch
    from jaero_b200 import synth
    fs = 2.048e6
    assert jb.channelizer_ratio(fs) == (3, 128)
    A = 300.0
    third = 1 / 3.0                                        # offsets on the 1/3 Hz grid keep the 3 s signal circular
    oq_off = [-690000 + 107000.0 * k + 1234 + (k % 3) * third for k in range(12)]
    strong_off = oq_off[5] + 25000.0
    ms_off = [-640000.0 + 2 * third, -210000.0 + 5555 + third, 305000.0 - 777, 655000.0 + 4321 + 2 * third]
    envs, sent, offs, amps, fbs = [], [], [], [], []
    for k, o in enumerate(oq_off + [strong_off]):
        bits, sus = _pchan_sus(10500, 6, 400 + k)
        envs.append(synth.oqpsk_envelope(bits, 10500)); sent.append(sus); offs.append(o)
        amps.append(A * (10 ** 1.5 if k == 12 else 1.0)); fbs.append(10500.0)
    for k, o in enumerate(ms_off):
        bits, sus = _pchan_sus(1200, 3, 500 + k)
        envs.append(synth.msk_envelope(bits, 1200)); sent.append(sus); offs.append(o)
        amps.append(A * np.sqrt(1200 / 10500.0)); fbs.append(1200.0)
    iq1 = synth.wideband_iq(envs, offs, fs, amplitudes=amps, ebn0_db=10.0, fb=fbs, seed=19, noise_ref=0, iq_format="cu8")
    assert len(iq1) == 3 * int(fs)
    iq = np.concatenate([iq1, iq1])
    d_iq = _dev(iq)
    modes = [("oqpsk", 10500, 12000.0, 1.0, list(range(13)), dict(lockingbw=10500.0)),
             ("msk", 1200, 3000.0, 8.0, list(range(13, 17)), dict(lockingbw=1800.0))]
    runs = []
    for kind, fb, pb, gain, idx, kw in modes:
        s = torch.cuda.Stream()
        ch = jb.Channelizer([offs[i] for i in idx], fs, passband_hz=pb, gain=gain, iq_format="cu8")
        b = jb.DemodBatch(kind, len(idx), fb=fb, freq_center=12000.0, **kw)
        pc = jb.PChannelBatch(len(idx), fb)
        ch.set_stream(s.cuda_stream); b.set_stream(s.cuda_stream)
        runs.append(dict(kind=kind, fb=fb, idx=idx, ch=ch, b=b, pc=pc, got=[[] for _ in idx], kw=kw, pb=pb, gain=gain))
    step = int(fs) // 4
    for k, a in enumerate(range(0, len(iq), step)):
        for r in runs:
            r["ch"].write_device(d_iq.data_ptr() + a * 2, min(step, len(iq) - a))
            p, n, st = r["ch"].output_device()
            r["b"].write_device(p, n, st)
            r["pc"].process_batch(r["b"])
            if k % 2 == 1:
                for c, v in enumerate(r["pc"].read_sus()):
                    r["got"][c].append(v)
    for r in runs:
        for c, v in enumerate(r["pc"].read_sus()):
            r["got"][c].append(v)
        dcd, _, _ = r["pc"].stats()
        assert np.all(dcd == 1), (r["kind"], dcd)
        for c, i in enumerate(r["idx"]):
            sus = np.concatenate([g[0] for g in r["got"][c]]); ok = np.concatenate([g[1] for g in r["got"][c]])
            good = {bytes(x) for x in sent[i].reshape(-1, 12)}
            valid = sus[ok == 1]
            assert len(valid) > 0, (r["kind"], c)
            assert all(bytes(x) in good for x in valid), (r["kind"], c)
        r["ok"] = [int(sum(g[1].sum() for g in r["got"][c])) for c in range(len(r["idx"]))]
    # the oracle chain on the float64 definition's audio of the same IQ: the weak carrier next to the strong one, one MSK
    x = iq_to_complex(iq, "cu8")
    for r, c in ((runs[0], 5), (runs[1], 0)):
        h = jb.channelizer_taps(fs, passband_hz=r["pb"])
        pcm = chan_poly_ref(x, h, 3, 128, [offs[r["idx"][c]]], fs, gain=r["gain"])[0]
        okw = dict(r["kw"], fft_power=14 if r["kind"] == "oqpsk" else 13, signalthreshold=0.65 if r["kind"] == "oqpsk" else 0.5)
        _, ok_o = _decode_oracle(r["kind"], pcm, r["fb"], okw)
        assert r["ok"][c] >= 0.95 * int(ok_o.sum()), (r["kind"], r["ok"][c], int(ok_o.sum()))
    for r in runs:
        r["ch"].close(); r["b"].close(); r["pc"].close()
