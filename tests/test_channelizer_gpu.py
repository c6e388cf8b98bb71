"""Device channelizer on the GPU: against the float64 definition (tests/chan_ref.py), independence from how the input is cut
into writes and from where a channel sits in the tile, selectivity, and wideband IQ through channelizer -> demodulator ->
P-channel layer to CRC-valid signal units."""
import numpy as np
import pytest

from chan_ref import chan_ref, iq_to_complex
from conftest import has_cuda

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not has_cuda(), reason="needs a CUDA device")]


def _jb():
    import jaero_b200
    return jaero_b200


def _dev(iq):
    import torch
    t = torch.from_numpy(np.ascontiguousarray(iq)).cuda()
    torch.cuda.synchronize()
    return t


def _noise_and_carriers(rng, n, fs, iq_format, n_car=5, noise=2500.0, amp=4000.0):
    t = np.arange(n)
    x = rng.normal(0, noise, n) + 1j * rng.normal(0, noise, n)
    for f in rng.uniform(-0.45 * fs, 0.45 * fs, n_car):
        x += amp * np.exp(2j * np.pi * (f * t / fs + rng.uniform()))
    a = np.stack([x.real, x.imag], axis=1)
    if iq_format == "cs16":
        return np.clip(np.rint(a), -32768, 32767).astype(np.int16)
    return np.clip(np.rint(a / 256.0 + 127.5), 0, 255).astype(np.uint8)


def _offsets(rng, C, fs, pb):
    edge = fs / 2 - pb / 2
    off = rng.uniform(-edge, edge, C)
    off[0], off[1], off[2] = edge, -edge, 0.0
    off[3:8] = -np.abs(off[3:8])
    return off


CASES = [  # iq_format, input_rate, output_rate, audio_hz, passband_hz
    ("cs16", 32 * 48000.0, 48000.0, 12000.0, 12000.0),
    ("cu8", 50 * 48000.0, 48000.0, 12000.0, 3000.0),
    ("cs16", 37 * 48000.0, 48000.0, 12000.0, 10000.0),
    ("cu8", 37 * 48000.0, 48000.0, 12000.0, 12000.0),
    ("cs16", 64 * 24000.0, 24000.0, 6000.0, 3000.0),
    ("cu8", 100 * 12000.0, 12000.0, 3000.0, 3000.0),
]


@pytest.mark.parametrize("case", CASES, ids=["%s-%d-%d" % (c[0], c[1] // c[2], c[2]) for c in CASES])
def test_channelizer_matches_reference(case):
    jb = _jb()
    fmt, fs, fo, audio, pb = case
    D = int(round(fs / fo))
    rng = np.random.default_rng(D * 7 + len(fmt))
    C = 70
    off = _offsets(rng, C, fs, pb)
    n = 700 * D + 13
    iq = _noise_and_carriers(rng, n, fs, fmt)
    ch = jb.Channelizer(off, fs, output_rate=fo, audio_hz=audio, passband_hz=pb, iq_format=fmt, gain=0.8)
    ch.write(iq)
    got = ch.read()
    h = jb.channelizer_taps(fs, output_rate=fo, audio_hz=audio, passband_hz=pb)
    want = chan_ref(iq_to_complex(iq, fmt), h, off, fs, output_rate=fo, audio_hz=audio, gain=0.8)
    assert got.shape == want.shape == (C, (n + D - 1) // D)
    d = np.abs(got.astype(np.int32) - want)
    assert d.max() <= 1, np.unravel_index(np.argmax(d), d.shape)
    assert np.mean(d == 0) >= 0.99, np.mean(d == 0)
    assert np.abs(want).max() > 1000                      # the comparison covers large values, not only noise
    ch.close()


def test_chunking_and_device_feed_are_bit_identical():
    jb = _jb()
    fs, D = 50 * 48000.0, 50
    rng = np.random.default_rng(5)
    off = _offsets(rng, 70, fs, 12000.0)
    n = 300 * D + 29
    iq = _noise_and_carriers(rng, n, fs, "cs16")
    one = jb.Channelizer(off, fs)
    one.write(iq)
    ref = one.read()
    sizes = [1, 2, D - 1, D, D + 1, 4097]
    cuts = np.cumsum(sizes)
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
    assert any(g.shape[1] == 0 for g in got)               # writes shorter than D can end without an output
    got, got_dev = np.concatenate(got, axis=1), np.concatenate(got_dev, axis=1)
    assert np.array_equal(got, ref)
    assert np.array_equal(got_dev, ref)
    assert many.launches >= 2 * len(pieces) - 3
    for c in (one, many, dev):
        c.close()


def test_rows_do_not_depend_on_position():
    jb = _jb()
    fs = 32 * 48000.0
    base = np.array([-701234.25, -3000.5, 17.0, 650001.75])
    off = np.tile(base, 256)                               # 1024 channels, 4 interleaved offsets
    rng = np.random.default_rng(11)
    iq = _noise_and_carriers(rng, 400 * 32 + 5, fs, "cs16")
    ch = jb.Channelizer(off, fs)
    ch.write(iq)
    out = ch.read()
    for c in range(4):
        assert np.array_equal(out[c::4], np.broadcast_to(out[c], out[c::4].shape)), c
    ch.close()


def _amp(row):
    return np.sqrt(2.0) * np.sqrt(np.mean(row.astype(np.float64) ** 2))


def test_selectivity_with_tones():
    jb = _jb()
    fs, D, pb, audio = 50 * 48000.0, 50, 12000.0, 12000.0
    fp = pb / 2
    f_s = min(2 * audio, 48000.0 - 2 * audio) - fp
    centre = 123456.0
    A, gain = 20000.0, 1.5
    deltas = [0.99 * fp, -0.99 * fp, f_s, -f_s, 1.5 * f_s, -3 * f_s, 100000.0, -400000.0]
    n = 4000 * D
    t = np.arange(n)
    rows = []
    for k, dlt in enumerate(deltas):                       # one tone at a time; every row sees the same tone
        x = A * np.exp(2j * np.pi * (centre + dlt) * t / fs)
        iq = np.clip(np.rint(np.stack([x.real, x.imag], axis=1)), -32768, 32767).astype(np.int16)
        c1 = jb.Channelizer([centre], fs, passband_hz=pb, gain=gain)
        c1.write(iq)
        rows.append(c1.read()[0, 100:])                   # past the filter's start-up (T = 727 < 100 D)
        c1.close()
    full = gain * A
    for dlt, r in zip(deltas[:2], rows[:2]):
        db = 20 * np.log10(_amp(r) / full)
        assert abs(db) <= 0.05, (dlt, db)
    for dlt, r in zip(deltas[2:], rows[2:]):
        a = _amp(r)
        assert a >= 0 and 20 * np.log10(max(a, 1e-9) / full) <= -58.0, (dlt, a)
    assert _amp(rows[2]) > 10.0                            # the suppressed tone is still tens of LSB, not rounded away


def _pchan_sus(fb, n_frames, seed):
    from jaero_b200 import synth
    return synth.pchannel_bits(fb, n_frames, seed, return_sus=True, loop=True, even_parity=(fb != 10500))


def test_device_feed_equals_host_feed():
    jb = _jb()
    import torch
    from jaero_b200 import synth
    fs = 32 * 48000.0
    offs = [-300000.0 + 1 / 3.0, 150000.0 + 2 / 3.0, 420000.0]
    envs = []
    for k in range(3):
        bits, _ = _pchan_sus(10500, 6, 70 + k)
        envs.append(synth.oqpsk_envelope(bits, 10500))
    iq = synth.wideband_iq(envs, offs, fs, amplitudes=[400.0] * 3, ebn0_db=12.0, fb=10500.0, seed=3)
    d_iq = _dev(iq)
    s = torch.cuda.Stream()
    ch = jb.Channelizer(offs, fs)
    ch.set_stream(s.cuda_stream)
    bd = jb.DemodBatch("oqpsk", 3, fb=10500, freq_center=12000.0)
    bd.set_stream(s.cuda_stream)
    bh = jb.DemodBatch("oqpsk", 3, fb=10500, freq_center=12000.0)
    step = 48000 * 32 // 4
    soft_d, soft_h = [[] for _ in range(3)], [[] for _ in range(3)]
    for a in range(0, len(iq), step):
        ch.write_device(d_iq.data_ptr() + a * 4, min(step, len(iq) - a))
        p, n, st = ch.output_device()
        bd.write_device(p, n, st)
        bh.write(ch.read())
        for c, v in enumerate(bd.read_softbits()):
            soft_d[c].append(v)
        for c, v in enumerate(bh.read_softbits()):
            soft_h[c].append(v)
    for c in range(3):
        a, b = np.concatenate(soft_d[c]), np.concatenate(soft_h[c])
        assert len(a) > 10000 and np.array_equal(a, b)
    ch.close(); bd.close(); bh.close()


def _decode_oracle(kind, pcm, fb, kw):
    from oracle import restated
    od = restated.OracleDemod(kind, fb=fb, freq_center=12000.0, **kw)
    op = restated.OraclePChannel(fb)
    for a in range(0, len(pcm), 4800):
        od.set_dcd(op.dcd)
        od.write(pcm[a:a + 4800])
        op.process(od.take_soft())
    b, ok, _ = op.take_sus()
    return b, ok


def test_wideband_iq_to_signal_units():
    """1.536 MHz cs16, 6 s (two loops of 3 s): 13 OQPSK 10.5k carriers (one of them 30 dB stronger, 25 kHz from a weak one)
    and 4 MSK 1200 carriers at Eb/N0 10 dB, two handles on the same device IQ, each with its own stream, batch and
    P-channel layer."""
    jb = _jb()
    import torch
    from jaero_b200 import synth
    fs = 32 * 48000.0
    A = 300.0
    third = 1 / 3.0                                        # offsets on the 1/3 Hz grid keep the 3 s signal circular
    oq_off = [-690000 + 107000.0 * k + 1234 + (k % 3) * third for k in range(12)]
    strong_off = oq_off[5] + 25000.0
    ms_off = [-640000.0 + 2 * third, -210000.0 + 5555 + third, 305000.0 - 777, 655000.0 + 4321 + 2 * third]
    envs, sent, offs, amps, fbs = [], [], [], [], []
    for k, o in enumerate(oq_off + [strong_off]):
        bits, sus = _pchan_sus(10500, 6, 200 + k)
        envs.append(synth.oqpsk_envelope(bits, 10500)); sent.append(sus); offs.append(o)
        amps.append(A * (10 ** 1.5 if k == 12 else 1.0)); fbs.append(10500.0)
    for k, o in enumerate(ms_off):
        bits, sus = _pchan_sus(1200, 3, 300 + k)
        envs.append(synth.msk_envelope(bits, 1200)); sent.append(sus); offs.append(o)
        amps.append(A * np.sqrt(1200 / 10500.0)); fbs.append(1200.0)
    iq1 = synth.wideband_iq(envs, offs, fs, amplitudes=amps, ebn0_db=10.0, fb=fbs, seed=9, noise_ref=0)
    iq = np.concatenate([iq1, iq1])
    d_iq = _dev(iq)
    modes = [("oqpsk", 10500, 12000.0, 1.0, list(range(13)), dict(lockingbw=10500.0)),
             ("msk", 1200, 3000.0, 8.0, list(range(13, 17)), dict(lockingbw=1800.0))]
    runs = []
    for kind, fb, pb, gain, idx, kw in modes:
        s = torch.cuda.Stream()
        ch = jb.Channelizer([offs[i] for i in idx], fs, passband_hz=pb, gain=gain)
        b = jb.DemodBatch(kind, len(idx), fb=fb, freq_center=12000.0, **kw)
        pc = jb.PChannelBatch(len(idx), fb)
        ch.set_stream(s.cuda_stream); b.set_stream(s.cuda_stream)
        runs.append(dict(kind=kind, fb=fb, idx=idx, ch=ch, b=b, pc=pc, got=[[] for _ in idx], kw=kw, pb=pb, gain=gain))
    step = int(fs) // 4
    for k, a in enumerate(range(0, len(iq), step)):
        for r in runs:
            r["ch"].write_device(d_iq.data_ptr() + a * 4, min(step, len(iq) - a))
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
    x = iq_to_complex(iq, "cs16")
    for r, c in ((runs[0], 5), (runs[1], 0)):
        h = jb.channelizer_taps(fs, passband_hz=r["pb"])
        pcm = chan_ref(x, h, [offs[r["idx"][c]]], fs, gain=r["gain"])[0]
        okw = dict(r["kw"], fft_power=14 if r["kind"] == "oqpsk" else 13, signalthreshold=0.65 if r["kind"] == "oqpsk" else 0.5)
        _, ok_o = _decode_oracle(r["kind"], pcm, r["fb"], okw)
        assert r["ok"][c] >= 0.95 * int(ok_o.sum()), (r["kind"], r["ok"][c], int(ok_o.sum()))
    for r in runs:
        r["ch"].close(); r["b"].close(); r["pc"].close()
