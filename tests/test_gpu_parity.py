"""GPU parity tests (pytest -m gpu, run on the B200 box): the CUDA path behind the C ABI against the CPU
oracle on the same inputs. Integer/byte outputs (soft bits after hard decision, Viterbi bits, SU bytes, CRC
flags) must be bit-exact; floating-point loop state within 1e-6 relative (north_star allows 1e-4)."""
import hashlib
import os

import numpy as np
import pytest

from conftest import ROOT, has_cuda, load_excerpt
from oracle import restated

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not has_cuda(), reason="needs a CUDA device")]
STATE_TOL = 1e-6


def _import():
    import jaero_b200
    return jaero_b200


def _interleave(soft, cols):
    n = soft.shape[-1]
    k = np.arange(n); i = k % 64; j = k // 64
    out = np.zeros_like(soft)
    out[..., ((i * 27) % 64) * cols + j] = soft[..., k]
    return out


def _noisy_code(rng, n, sigma):
    msg = rng.integers(0, 256, size=n // 16, dtype=np.uint8)
    enc = restated.conv_encode(msg)[:n].astype(np.float64)
    x = (enc * 2 - 1) * 60 + 128 + rng.normal(0, sigma, size=n)
    return msg, np.clip(np.round(x), 0, 255).astype(np.uint8)


@pytest.mark.parametrize("cols", [78, 9, 6])
def test_viterbi_continuous_bit_exact(cols):
    jb = _import()
    rng = np.random.default_rng(cols)
    C, n = 7, 64 * cols
    vb = jb.ViterbiBatch(C, 24)
    orc = [restated.OracleViterbi(24) for _ in range(C)]
    for it in range(4):
        soft = np.stack([_noisy_code(rng, n, 30 + 12 * c)[1] for c in range(C)])
        if it == 2:
            soft[0] = rng.integers(0, 256, size=n, dtype=np.uint8)     # pure noise: exercises ties / renormalisation
            soft[1] = 128                                               # all erasures
        got = vb.decode_continuous(_interleave(soft, cols), cols)
        for c in range(C):
            ref = orc[c].decode_continuous(soft[c]).astype(np.uint8)
            assert vb.last_valid[c] == len(ref)
            assert np.array_equal(ref, got[c][:len(ref)]), (it, c)
    vb.reset()
    fresh = restated.OracleViterbi(24)
    soft = np.stack([_noisy_code(rng, n, 40)[1]] * C)
    got = vb.decode_continuous(soft, 0)
    ref = fresh.decode_continuous(soft[0]).astype(np.uint8)
    assert all(np.array_equal(ref, got[c][:len(ref)]) for c in range(C))


def test_viterbi_block_decode_and_edge_sizes():
    jb = _import()
    rng = np.random.default_rng(9)
    for n in (32, 64, 600, 1234 * 2):
        C = 5
        vb = jb.ViterbiBatch(C, 24)
        blk = rng.integers(0, 256, size=(C, n), dtype=np.uint8)
        got = vb.decode_block(blk)
        for c in range(C):
            ref = restated.conv_decode_soft(blk[c])[:n // 2 - 6]
            assert np.array_equal(ref, got[c][:n // 2 - 6])
        with pytest.raises(jb.JaeroError):
            vb.decode_block(blk[:, :31])
        vb.close()


def test_viterbi_full_size_roundtrip_property():
    """4096 channels x 4992 soft values (BASELINE cfg 3 block size): encode -> AWGN -> decode recovers the message."""
    jb = _import()
    rng = np.random.default_rng(1)
    C, n = 4096, 4992
    base = [_noisy_code(rng, n, 35) for _ in range(16)]
    idx = rng.integers(0, 16, size=C)
    soft = np.stack([base[i][1] for i in idx])
    vb = jb.ViterbiBatch(C, 24)
    got = vb.decode_continuous(soft, 0)
    for c in range(0, C, 37):
        bits = np.unpackbits(base[idx[c]][0])
        # first call: output bit j = trellis bit 25+j  (no overlap prefix)
        assert np.array_equal(got[c][:2400], bits[25:2425])
    assert len({hashlib.sha256(got[c].tobytes()).hexdigest() for c in range(C)}) <= 16   # identical inputs -> identical outputs


def _run_gpu(kind, pcm2, kw, chunk, dcd_sched=None, read_every=8, **extra):
    jb = _import()
    b = jb.DemodBatch(kind, pcm2.shape[0], **kw, **extra)
    acc = [[] for _ in range(pcm2.shape[0])]
    sched = dict(dcd_sched or [])
    for k, a in enumerate(range(0, pcm2.shape[1], chunk)):
        if a in sched:
            b.set_dcd(sched[a])
        b.write(pcm2[:, a:a + chunk])
        if k % read_every == read_every - 1:
            for c, s in enumerate(b.read_softbits()):
                acc[c].append(s)
    for c, s in enumerate(b.read_softbits()):
        acc[c].append(s)
    st = b.status()
    b.close()
    return [np.concatenate(x) for x in acc], st


def _run_oracle(kind, pcm, kw, chunk, dcd_sched=None):
    d = restated.OracleDemod(kind, **kw)
    sched = dict(dcd_sched or [])
    for a in range(0, len(pcm), chunk):
        if a in sched:
            d.set_dcd(sched[a])
        d.write(pcm[a:a + chunk])
    return d.take_soft(), d.state()


def _assert_parity(soft_g, st_g, soft_o, st_o):
    assert len(soft_g) == len(soft_o)
    assert np.array_equal(soft_g >= 128, soft_o >= 128)                  # bit-exact after hard decision
    assert np.abs(soft_g.astype(int) - soft_o.astype(int)).max(initial=0) <= 1   # soft bytes: at most 1 LSB (libm ulp)
    for k, v in st_o.items():
        if k in st_g and k not in ("n_sig_true", "n_sig_false"):
            assert abs(st_g[k] - v) <= STATE_TOL * max(abs(v), 1e-9) + 1e-12, (k, st_g[k], v)
    assert st_g["n_sig_true"] == st_o["n_sig_true"] and st_g["n_sig_false"] == st_o["n_sig_false"]


@pytest.mark.parametrize("name", ["oqpsk_10500", "oqpsk_10500_noafc_dcd", "oqpsk_8400", "msk_600", "msk_1200", "msk_1200_noafc_dcd"])
def test_demod_parity_on_reference_recordings(golden, name):
    case = golden[name]
    pcm = load_excerpt(case["excerpt"])
    pcm2 = np.stack([pcm, (pcm.astype(np.int32) * 2 // 3).astype(np.int16), pcm[::-1].copy()])
    kw = dict(case["kw"])
    sched = [(int(a), int(v)) for a, v in case["dcd_schedule"]]
    soft_g, st_g = _run_gpu(case["kind"], pcm2, kw, case["chunk"], sched)
    for c in range(3):
        soft_o, st_o = _run_oracle(case["kind"], pcm2[c], kw, case["chunk"], sched)
        _assert_parity(soft_g[c], st_g[c], soft_o, st_o)
    # channel 0 is the committed golden produced by the verbatim reference build
    assert len(soft_g[0]) == case["n_soft"]
    if hashlib.sha256(soft_g[0].astype("<i2").tobytes()).hexdigest() != case["soft_sha256"]:
        # The only admissible difference from the verbatim reference's stream: isolated soft values one LSB off (a libm call
        # rounding the other way just at a quantiser step; never across 127/128, that was asserted above). The restated oracle
        # IS sha-identical to the golden (tests/test_oracle_golden.py), so the indices can be listed against it.
        soft_o, _ = _run_oracle(case["kind"], pcm2[0], kw, case["chunk"], sched)
        assert hashlib.sha256(soft_o.astype("<i2").tobytes()).hexdigest() == case["soft_sha256"]
        diff = np.nonzero(soft_g[0] != soft_o)[0]
        assert len(diff) <= max(2, len(soft_o) // 5000), "too many soft values differ from the reference: %s" % diff[:20]
        assert np.abs(soft_g[0][diff].astype(int) - soft_o[diff].astype(int)).max() == 1
        print("golden %s: %d of %d soft values one LSB off the verbatim reference at indices %s" % (name, len(diff), len(soft_o), diff.tolist()))


@pytest.mark.parametrize("ebn0", [6.0, 8.0, 10.0, None])
def test_oqpsk_parity_synthetic_ebn0_sweep(ebn0):
    """BASELINE cfg 3 signal model (P-channel OQPSK 10.5k, Eb/N0 sweep): identical hard decisions, hence identical BER."""
    from jaero_b200 import synth
    chans = []
    for c in range(4):
        chans.append(synth.oqpsk_pchannel_pcm(6, fc=8000.0 + 37.0 * c, seed=100 + c, ebn0_db=ebn0, phase=0.7 * c, delay=3 * c))
    pcm2 = np.stack(chans)
    kw = dict(fb=10500, freq_center=8000.0, lockingbw=10500, fft_power=14, signalthreshold=0.65, afc=False)
    soft_g, st_g = _run_gpu("oqpsk", pcm2, kw, 6000)
    for c in range(4):
        soft_o, st_o = _run_oracle("oqpsk", pcm2[c], kw, 6000)
        _assert_parity(soft_g[c], st_g[c], soft_o, st_o)
    assert sum(len(s) for s in soft_g) > 10000


def test_msk1200_parity_synthetic_cfg2():
    """BASELINE cfg 2 signal model (continuous 1200 bps MSK P-channel, Eb/N0 = 8 dB, carriers 2000 +- 200 Hz, random phase and
    timing): soft bits / loop state against the oracle, then the device P-channel layer against the oracle's, DCD fed back on
    both sides at the same boundaries (DCD switches the MSK timing-loop gain, mskdemodulator.cpp:387-405)."""
    jb = _import()
    from jaero_b200 import synth
    C = 5
    fcs = [2000.0, 1831.0, 2177.0, 2064.5, 1950.25]
    pcm2 = np.stack([np.tile(synth.msk_pchannel_pcm(4, fc=fcs[c], seed=500 + c, ebn0_db=8.0, fb=1200.0, phase=1.3 * c, delay=7 * c), 3) for c in range(C)])
    kw = dict(fb=1200, freq_center=2000.0, lockingbw=1800, fft_power=13, signalthreshold=0.5, afc=False)
    soft_g, st_g = _run_gpu("msk", pcm2, kw, 6000)
    for c in range(C):
        soft_o, st_o = _run_oracle("msk", pcm2[c], kw, 6000)
        _assert_parity(soft_g[c], st_g[c], soft_o, st_o)
    assert all(len(s) == len(soft_g[0]) for s in soft_g) and len(soft_g[0]) > 12000
    # demodulator + frame layer with the DCD loop closed
    b = jb.DemodBatch("msk", C, **kw)
    pc = jb.PChannelBatch(C, 1200)
    od = [restated.OracleDemod("msk", **kw) for _ in range(C)]
    op = [restated.OraclePChannel(1200) for _ in range(C)]
    got = [[] for _ in range(C)]
    for k, a in enumerate(range(0, pcm2.shape[1], 4800)):
        b.write(pcm2[:, a:a + 4800]); pc.process_batch(b)
        for c in range(C):
            od[c].set_dcd(op[c].dcd); od[c].write(pcm2[c, a:a + 4800]); op[c].process(od[c].take_soft())
        if k % 10 == 9:
            pc.tick(b)
            for c in range(C):
                op[c].update_dcd()
            for c, r in enumerate(pc.read_sus()):
                got[c].append(r)
    for c, r in enumerate(pc.read_sus()):
        got[c].append(r)
    st = b.status()
    for c in range(C):
        gb = np.concatenate([g[0] for g in got[c]]); gok = np.concatenate([g[1] for g in got[c]])
        rb, rok, _ = op[c].take_sus()
        assert np.array_equal(gb, rb) and np.array_equal(gok, rok)
        o = od[c].state()
        for key in ("mixer2_freq", "st_wtptr", "mse", "agc"):
            scale = 19999.0 if key.endswith("wtptr") else max(abs(o[key]), 1e-9)   # a table pointer is a phase: error relative to one cycle
            assert abs(st[c][key] - o[key]) <= STATE_TOL * scale, key
    assert sum(int(np.concatenate([g[1] for g in got[c]]).sum()) for c in range(C)) >= 40 * C // 2
    b.close(); pc.close()


def test_msk1200_full_size_batch_consistency():
    """BASELINE cfg 2 size (1024 channels): channels fed the same stream agree whatever warp / CTA they sit in, and match the oracle."""
    from jaero_b200 import synth
    C = 1024
    variants = np.stack([synth.msk_pchannel_pcm(3, fc=1900.0 + 70 * v, seed=900 + v, ebn0_db=8.0, fb=1200.0, phase=0.9 * v, delay=11 * v) for v in range(4)])
    idx = (np.arange(C) * 7 + np.arange(C) // 32) % 4
    pcm2 = np.ascontiguousarray(variants[idx])
    kw = dict(fb=1200, freq_center=2000.0, lockingbw=1800, fft_power=13, signalthreshold=0.5, afc=True)
    soft, st = _run_gpu("msk", pcm2, kw, 9999, read_every=2)
    for v in range(4):
        members = np.nonzero(idx == v)[0]
        assert all(np.array_equal(soft[members[0]], soft[m]) for m in members[1:])
        assert len({st[m]["mixer2_wtptr"] for m in members}) == 1 and len({st[m]["mse"] for m in members}) == 1
        so, sto = _run_oracle("msk", variants[v], kw, 9999)
        _assert_parity(soft[members[0]], st[members[0]], so, sto)


def test_chunking_and_settings_variants():
    """writeData results do not depend on how the stream is chunked; cpu_reduce / sql / no-EbNo variants match the oracle."""
    pcm = load_excerpt("oqpsk_10500")[:48000 * 5]
    base = dict(fb=10500, freq_center=5760, lockingbw=10500, fft_power=14, signalthreshold=0.65)
    pcm2 = np.stack([pcm, pcm])
    a, sa = _run_gpu("oqpsk", pcm2, dict(base, afc=True), 4800)
    b, sb = _run_gpu("oqpsk", pcm2, dict(base, afc=True), 7777, read_every=3)
    c, sc = _run_gpu("oqpsk", pcm2, dict(base, afc=True), 333, read_every=40)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[0], c[0]) and np.array_equal(a[0], a[1])
    assert sa[0]["mixer2_wtptr"] == sb[0]["mixer2_wtptr"] == sc[0]["mixer2_wtptr"]
    for variant in (dict(cpureduce=True), dict(sql=True), dict(afc=True, fft_power=13)):
        kw = dict(base); kw.update({k: v for k, v in variant.items() if k != "cpureduce"})
        gk = dict(kw); ok_ = dict(kw)
        if "cpureduce" in variant:
            gk["cpu_reduce"] = True; ok_["cpureduce"] = True
        soft_g, st_g = _run_gpu("oqpsk", pcm2[:1], gk, 4800)
        soft_o, st_o = _run_oracle("oqpsk", pcm, ok_, 4800)
        _assert_parity(soft_g[0], st_g[0], soft_o, st_o)
    # EbNo observable off: data path unchanged
    d, sd = _run_gpu("oqpsk", pcm2[:1], dict(base, afc=True), 4800, report_ebno=False)
    assert np.array_equal(d[0], a[0]) and sd[0]["ebno"] == 0.0


def test_ragged_channel_count_and_lane_consistency():
    """A channel count that is not a multiple of 32: every channel fed the same stream must produce the same output."""
    pcm = load_excerpt("oqpsk_10500")[:48000 * 3]
    C = 70
    pcm2 = np.ascontiguousarray(np.broadcast_to(pcm, (C, len(pcm))))
    soft, st = _run_gpu("oqpsk", pcm2, dict(fb=10500, freq_center=5760, lockingbw=10500, afc=True), 4096)
    assert all(np.array_equal(soft[0], s) for s in soft)
    assert len({s["mixer2_wtptr"] for s in st}) == 1
    soft_o, st_o = _run_oracle("oqpsk", pcm, dict(fb=10500, freq_center=5760, lockingbw=10500, fft_power=14, signalthreshold=0.65, afc=True), 4096)
    _assert_parity(soft[C - 1], st[C - 1], soft_o, st_o)


def test_full_size_batch_consistency():
    """BASELINE cfg 3 size (4096 channels): channels that receive the same stream produce identical soft bits and loop
    state whatever warp / block / staging tile they sit in, and match the oracle."""
    pcm = load_excerpt("oqpsk_10500")[:48000 * 2 + 1234]
    C = 4096
    variants = np.stack([pcm, (pcm.astype(np.int32) * 2 // 3).astype(np.int16), pcm[::-1].copy(), np.roll(pcm, 777)])
    idx = np.arange(C) % 4
    pcm2 = np.ascontiguousarray(variants[idx])
    soft, st = _run_gpu("oqpsk", pcm2, dict(fb=10500, freq_center=5760, lockingbw=10500, afc=True), 9999, read_every=2)
    for v in range(4):
        members = np.nonzero(idx == v)[0]
        ref_soft = soft[members[0]]
        assert all(np.array_equal(ref_soft, soft[m]) for m in members[1:])
        assert len({st[m]["mixer2_wtptr"] for m in members}) == 1 and len({st[m]["mse"] for m in members}) == 1
        so, sto = _run_oracle("oqpsk", variants[v], dict(fb=10500, freq_center=5760, lockingbw=10500, fft_power=14, signalthreshold=0.65, afc=True), 9999)
        _assert_parity(ref_soft, st[members[0]], so, sto)


def test_pchannel_frame_layer_bit_exact(golden):
    """Device framing + fused de-interleave/Viterbi + descramble + CRC == restated AeroL::Decode on the same soft bits,
    with DCD fed back to the demodulators at chunk boundaries on both sides."""
    jb = _import()
    for name in ("oqpsk_10500", "msk_600"):
        case = golden[name]
        kind, kw = case["kind"], dict(case["kw"])
        pcm = load_excerpt(case["excerpt"])
        pcm2 = np.stack([pcm, (pcm.astype(np.int32) * 3 // 4).astype(np.int16)])
        b = jb.DemodBatch(kind, 2, **kw)
        pc = jb.PChannelBatch(2, kw["fb"])
        od = [restated.OracleDemod(kind, **kw) for _ in range(2)]
        op = [restated.OraclePChannel(kw["fb"]) for _ in range(2)]
        got = [[], []]
        chunk = 4096
        for k, a in enumerate(range(0, pcm2.shape[1], chunk)):
            b.write(pcm2[:, a:a + chunk]); pc.process_batch(b)
            for c in range(2):
                od[c].set_dcd(op[c].dcd); od[c].write(pcm2[c, a:a + chunk]); op[c].process(od[c].take_soft())
            if k % 11 == 10:
                for c, r in enumerate(pc.read_sus()):
                    got[c].append(r)
            if (a + chunk) % 48000 < chunk:
                pc.tick(b)
                for c in range(2):
                    op[c].update_dcd()
        for c, r in enumerate(pc.read_sus()):
            got[c].append(r)
        dcd, tot, okc = pc.stats()
        for c in range(2):
            gb = np.concatenate([g[0] for g in got[c]]); gok = np.concatenate([g[1] for g in got[c]])
            rb, rok, _ = op[c].take_sus()
            assert np.array_equal(gb, rb) and np.array_equal(gok, rok)
            assert dcd[c] == int(op[c].dcd) and tot[c] == len(rok) and okc[c] == rok.sum()
        assert int(np.concatenate([g[1] for g in got[0]]).sum()) == case["n_su_crc_ok"]      # golden from the verbatim reference
        b.close(); pc.close()


@pytest.mark.parametrize("name", ["burst_msk_1200_a", "burst_msk_1200_b", "burst_oqpsk_10500"])
def test_burst_parity_on_reference_recordings(golden, name):
    """BASELINE cfg 4 source material (burst MSK 1200) and the 10.5k burst OQPSK recording: Hilbert FFT-FIR, burst
    detector, trident FFT acquisition, preamble-aided tail. Soft bits (incl. the -1 start-of-burst markers) identical
    after hard decision and within 1 LSB; gain / carrier from the acquisition FFTs within 1e-6."""
    jb = _import()
    case = golden[name]
    pcm = load_excerpt(name)
    pcm2 = np.stack([pcm, (pcm.astype(np.int32) * 3 // 5).astype(np.int16), np.roll(pcm, 12345)])
    b = (jb.BurstOqpskBatch if case["kind"] == "burst_oqpsk" else jb.BurstMskBatch)(3, **case["kw"])
    acc = [[] for _ in range(3)]
    for a in range(0, pcm2.shape[1], case["chunk"]):
        b.write(pcm2[:, a:a + case["chunk"]])
        for c, s in enumerate(b.read_softbits()):
            acc[c].append(s)
    st = b.status()
    b.close()
    for c in range(3):
        o = restated.OracleDemod(case["kind"], **case["kw"])
        for a in range(0, pcm2.shape[1], case["chunk"]):
            o.write(pcm2[c, a:a + case["chunk"]])
        so = o.take_soft(); sg = np.concatenate(acc[c]); os_ = o.state()
        assert len(so) == len(sg)
        assert np.array_equal(so < 0, sg < 0) and np.array_equal(so >= 128, sg >= 128)
        assert np.abs(so.astype(int) - sg.astype(int)).max(initial=0) <= 1
        for k in ("mixer2_freq", "vol_gain", "mse", "agc", "st_wtptr", "rotator_freq"):
            assert abs(st[c][k] - os_[k]) <= STATE_TOL * max(abs(os_[k]), 1e-9), k
        for k in ("n_sig_true", "n_sig_false", "cntr", "startstop"):
            assert st[c][k] == os_[k], k
        eb = o.take_aux(0)
        assert st[c]["n_ebno_emits"] == len(eb) and (len(eb) == 0 or abs(st[c]["last_burst_ebno"] - eb[-1]) < 1e-6)
    assert len(np.concatenate(acc[0])) == case["n_soft"]          # golden from the verbatim reference build
    assert int((np.concatenate(acc[0]) < 0).sum()) >= 2


def test_burst_replicas_with_frequency_offsets_cfg4(golden):
    """BASELINE cfg 4 as specified: 32 replicas of samples/1200bps_burst_sample1.wav, replica r = Re{hilbert(x) e^(j 2 pi df_r n/Fs)},
    df_r = U(-300, 300) Hz from seed 0xB0057 + r. Every replica's acquisition lands on a different bin of the two 32768-point
    trident FFTs (burstmskdemodulator.cpp:443-568): start-of-burst markers, estimated carrier, gain and the hard-decided soft
    bits must equal the oracle's for each of them."""
    import multiprocessing as mp
    from jaero_b200 import synth
    jb = _import()
    case = golden["burst_msk_1200_a"]
    base = load_excerpt("burst_msk_1200_a")
    R = 32
    offs = synth.replica_offsets(0, R)
    assert len(set(np.round(offs).astype(int))) == R and np.abs(offs).max() <= 300
    reps = synth.offset_replicas(base, offs)
    b = jb.BurstMskBatch(R, **case["kw"])
    acc = [[] for _ in range(R)]
    for a in range(0, reps.shape[1], 48000):
        b.write(reps[:, a:a + 48000])
        for c, s in enumerate(b.read_softbits()):
            acc[c].append(s)
    st = b.status()
    b.close()
    with mp.get_context("spawn").Pool(min(16, os.cpu_count() or 1)) as pool:
        ref = pool.map(restated.run_demod_job, [("burst_msk", case["kw"], reps[r], 48000) for r in range(R)])
    carriers = set()
    for r in range(R):
        so, os_, eb = ref[r]
        sg = np.concatenate(acc[r])
        assert len(so) == len(sg), r
        assert np.array_equal(np.nonzero(so < 0)[0], np.nonzero(sg < 0)[0]), r          # -1 marker positions
        assert np.array_equal(so >= 128, sg >= 128), r
        assert np.abs(so.astype(int) - sg.astype(int)).max(initial=0) <= 1
        for k in ("mixer2_freq", "vol_gain", "rotator_freq", "mse"):
            assert abs(st[r][k] - os_[k]) <= STATE_TOL * max(abs(os_[k]), 1e-9), (r, k)
        for k in ("n_sig_true", "n_sig_false", "cntr", "startstop"):
            assert st[r][k] == os_[k], (r, k)
        assert st[r]["n_ebno_emits"] == len(eb)
        carriers.add(round(st[r]["mixer2_freq"], 1))
    assert len(carriers) >= R - 2                                  # the offsets really spread the acquisitions over the spectrum
    assert sum(int((np.concatenate(acc[r]) < 0).sum()) for r in range(R)) >= 2 * R


def test_c_channel_replicas_and_two_modes_on_two_streams_cfg5(golden):
    """BASELINE cfg 5 building blocks: (i) 8400 bps C-channel replicas with frequency offsets (the reference's recording,
    Hilbert-rotated) through K6 + K1a' + the C-channel layer == the oracle chain; (ii) a 10.5k batch and an 8400 batch of the
    same process written alternately (as bench.py --workload mix16384 does per rank) give what each gives alone."""
    from jaero_b200 import synth
    jb = _import()
    base = load_excerpt("oqpsk_8400")
    offs = synth.replica_offsets(0, 3, span_hz=200.0, seed0=0xC8400)
    reps = synth.offset_replicas(base, offs)
    kw8 = dict(golden["oqpsk_8400"]["kw"])
    kwp = dict(golden["oqpsk_10500"]["kw"])
    pcm_p = load_excerpt("oqpsk_10500")[:reps.shape[1]]
    pcm_p2 = np.stack([pcm_p, pcm_p[::-1].copy()])
    ref_p, _ = _run_gpu("oqpsk", pcm_p2, kwp, 4800)
    b8 = jb.DemodBatch("oqpsk", 3, **kw8); cc = jb.CChannelBatch(3)
    bp = jb.DemodBatch("oqpsk", 2, **kwp)
    got8 = [[] for _ in range(3)]; gotp = [[], []]
    for k, a in enumerate(range(0, reps.shape[1], 4800)):
        b8.write(reps[:, a:a + 4800]); bp.write(pcm_p2[:, a:a + 4800])
        cc.process_batch(b8)
        if k % 10 == 9:
            cc.tick(b8)
        for c, fr in enumerate(cc.read_frames()):
            got8[c].append(fr)
        if k % 8 == 7:
            for c, s_ in enumerate(bp.read_softbits()):
                gotp[c].append(s_)
    for c, s_ in enumerate(bp.read_softbits()):
        gotp[c].append(s_)
    b8.close(); cc.close(); bp.close()
    for c in range(2):
        assert np.array_equal(np.concatenate(gotp[c]), ref_p[c])
    total_ok = 0
    for c in range(3):
        o = restated.OracleDemod("oqpsk", **kw8); oc = restated.OracleCChannel()
        for k, a in enumerate(range(0, reps.shape[1], 4800)):
            o.write(reps[c, a:a + 4800])
            oc.process(o.take_soft())
            o.set_dcd(int(oc.dcd))
            if k % 10 == 9:
                oc.update_dcd(); o.set_dcd(int(oc.dcd))
        su, cok, voice = oc.take_frames()
        gsu = np.concatenate([g[0] for g in got8[c]]); gok = np.concatenate([g[1] for g in got8[c]]); gv = np.concatenate([g[2] for g in got8[c]])
        assert gsu.shape == su.shape and np.array_equal(gsu, su) and np.array_equal(gok, cok) and np.array_equal(gv, voice)
        total_ok += int(cok.sum())
    assert total_ok >= 20


@pytest.mark.parametrize("name", ["burst_msk_1200_a", "burst_msk_1200_b", "burst_oqpsk_10500"])
def test_rt_channel_packets_on_reference_recordings(golden, name):
    """SURVEY 8(f)2 end to end on the GPU: burst demodulator -> R/T packet layer (unique word, trial de-interleave + Viterbi
    at every candidate length, descramble, CRC-16) with the soft bits never leaving the device; packets, SU counts and the
    number of trial decodes identical to the restated oracle chain; channel 0 equals the committed golden."""
    jb = _import()
    case = golden[name]
    pcm = load_excerpt(name)
    pcm2 = np.stack([pcm, np.roll(pcm, 7001)])
    oq = case["kind"] == "burst_oqpsk"
    b = (jb.BurstOqpskBatch if oq else jb.BurstMskBatch)(2, **case["kw"])
    rt = jb.RTChannelBatch(2, case["kw"]["fb"])
    got = [[], []]
    for k, a in enumerate(range(0, pcm2.shape[1], case["chunk"])):
        b.write(pcm2[:, a:a + case["chunk"]])
        rt.process_burst(b)
        if k % 10 == 9:
            rt.tick()
        for c, pk in enumerate(rt.read_packets()):
            got[c] += pk
    tr, bad, dcd = rt.stats()
    b.close(); rt.close()
    for c in range(2):
        o = restated.OracleDemod(case["kind"], **case["kw"])
        ort = restated.OracleRTChannel(case["kw"]["fb"])
        for k, a in enumerate(range(0, pcm2.shape[1], case["chunk"])):
            o.write(pcm2[c, a:a + case["chunk"]])
            ort.process(o.take_soft())
            if k % 10 == 9:
                ort.update_dcd()
        ref = ort.packets()
        assert len(ref) == len(got[c]) and tr[c] == ort.trials
        for r, g in zip(ref, got[c]):
            assert r["type"] == g["type"] and r["nsus"] == g["nsus"] and np.array_equal(r["bytes"], g["bytes"])
    assert [hashlib.sha256(g["bytes"].tobytes()).hexdigest() for g in got[0]] == [q["sha256"] for q in case["rt_packets"]]


def test_c_channel_frames_on_reference_recording(golden):
    """SURVEY 8(f)3 end to end on the GPU: 8400 bps demodulator (K6 + K1a') -> C-channel frame layer with the soft bits
    and the DCD feedback staying on the device; signal units, CRC flags and voice bytes identical to the oracle chain."""
    jb = _import()
    case = golden["oqpsk_8400"]
    pcm = load_excerpt("oqpsk_8400")
    pcm2 = np.stack([pcm, (pcm.astype(np.int32) * 2 // 3).astype(np.int16)])
    kw = dict(case["kw"])
    b = jb.DemodBatch("oqpsk", 2, **kw)
    cc = jb.CChannelBatch(2)
    got = [[], []]
    for k, a in enumerate(range(0, pcm2.shape[1], 4800)):
        b.write(pcm2[:, a:a + 4800])
        cc.process_batch(b)
        if k % 10 == 9:
            cc.tick(b)
        for c, fr in enumerate(cc.read_frames()):
            got[c].append(fr)
    dcd, tot, okc = cc.stats()
    b.close(); cc.close()
    for c in range(2):
        o = restated.OracleDemod("oqpsk", **kw); oc = restated.OracleCChannel()
        for k, a in enumerate(range(0, pcm2.shape[1], 4800)):
            o.write(pcm2[c, a:a + 4800])
            oc.process(o.take_soft())
            o.set_dcd(int(oc.dcd))
            if k % 10 == 9:
                oc.update_dcd(); o.set_dcd(int(oc.dcd))
        su, cok, voice = oc.take_frames()
        gsu = np.concatenate([g[0] for g in got[c]]); gok = np.concatenate([g[1] for g in got[c]]); gv = np.concatenate([g[2] for g in got[c]])
        assert gsu.shape == su.shape and np.array_equal(gsu, su) and np.array_equal(gok, cok) and np.array_equal(gv, voice)
        assert dcd[c] == int(oc.dcd) and tot[c] == cok.size and okc[c] == cok.sum()
        if c == 0:
            assert len(su) >= 5 and int(cok.sum()) >= 10


@pytest.mark.parametrize("kind,name,kw", [
    ("oqpsk", "oqpsk_10500", dict(fb=10500, freq_center=5760, lockingbw=10500, fft_power=14, signalthreshold=0.65, afc=True)),
    ("msk", "msk_600", dict(fb=600, freq_center=1000, lockingbw=900, fft_power=13, signalthreshold=0.5, afc=True)),
])
def test_pipeline_kernels_with_tiny_and_odd_writes(kind, name, kw):
    """The warp-specialised segment kernels hand samples between warps through named barriers; writes of 1, 2, 3 ... samples
    (launches whose loop body runs 0, 1 or 2 times, estimator triggers on the first / last sample of a call) must give the
    same stream as regular 4800-sample writes."""
    jb = _import()
    pcm = load_excerpt(name)[:48000 * 3]
    pcm2 = np.stack([pcm, pcm[::-1].copy(), (pcm // 2).astype(np.int16)])
    ref, st_ref = _run_gpu(kind, pcm2, kw, 4800)
    b = jb.DemodBatch(kind, 3, **kw)
    acc = [[] for _ in range(3)]
    pattern = [1, 2, 3, 1, 5, 4093, 1, 1, 2, 4096, 7, 2047, 1, 2049, 31, 33, 4800, 64, 1]
    a = 0; k = 0
    while a < pcm2.shape[1]:
        n = min(pattern[k % len(pattern)], pcm2.shape[1] - a)
        b.write(pcm2[:, a:a + n]); a += n; k += 1
        if k % 6 == 0:
            for c, s_ in enumerate(b.read_softbits()):
                acc[c].append(s_)
    for c, s_ in enumerate(b.read_softbits()):
        acc[c].append(s_)
    st = b.status()
    b.close()
    for c in range(3):
        assert np.array_equal(np.concatenate(acc[c]), ref[c])
        for key in ("mixer2_freq", "mixer2_wtptr", "st_wtptr", "mse", "agc"):
            assert st[c][key] == st_ref[c][key], key


def test_ingest_router_feeds_a_batch_like_direct_writes():
    """Messages of uneven sizes per channel, flushed whenever every channel has data, give the same soft bits as write()."""
    import struct
    jb = _import()
    pcm = load_excerpt("oqpsk_10500")[:48000 * 3]
    pcm2 = np.stack([pcm, pcm[::-1].copy()])
    kw = dict(fb=10500, freq_center=5760, lockingbw=10500, fft_power=14, signalthreshold=0.65, afc=True)
    ref, _ = _run_gpu("oqpsk", pcm2, kw, 4800)
    b = jb.DemodBatch("oqpsk", 2, **kw)
    r = jb.IngestRouter(["CHAN0", "CHAN1"], 48000, capacity_samples=60000)
    rate = struct.pack("<I", 48000)
    pos = [0, 0]; sizes = [[4800, 1234, 9000], [7000, 4800, 333]]
    acc = [[], []]; k = 0
    while min(pos) < pcm2.shape[1]:
        for c in range(2):
            n = min(sizes[c][k % 3], pcm2.shape[1] - pos[c])
            if n:
                assert r.message(b"CHAN%d" % c, rate, pcm2[c, pos[c]:pos[c] + n].tobytes()) == c
                pos[c] += n
        k += 1
        if r.available:
            r.flush(b)
            for c, s_ in enumerate(b.read_softbits()):
                acc[c].append(s_)
    assert r.available == 0
    b.close(); r.close()
    for c in range(2):
        assert np.array_equal(np.concatenate(acc[c]), ref[c])


@pytest.mark.parametrize("fb", [1200, 10500])
def test_rt_channel_known_answer_r_packets(fb):
    """Known-answer R packets (both polarities, different payloads per channel) through the GPU R/T layer."""
    from conftest import synthetic_r_packet_stream
    jb = _import()
    payloads = [((np.arange(17) * (7 + 2 * c) + c) % 256).astype(np.uint8) for c in range(5)]
    streams = [synthetic_r_packet_stream(fb, payloads[c], invert=bool(c & 1)) for c in range(5)]
    rt = jb.RTChannelBatch(5, fb)
    for a in range(0, max(len(s_) for s_ in streams), 97):           # odd chunking: packets straddle calls
        rt.process([s_[a:a + 97] for s_ in streams])
    got = rt.read_packets()
    rt.close()
    for c in range(5):
        assert len(got[c]) == 1 and got[c][0]["type"] == 1
        assert np.array_equal(got[c][0]["bytes"][:17], payloads[c]) and len(got[c][0]["bytes"]) == 19


# The reference's demodulator on the committed first 12 s of the 10.5k recording, framed by the restated P-channel layer and
# reassembled by the reference's own code, gives exactly the first 520 CRC-valid signal units and the first 11 records (6 of
# them ACARS) of what it gives on the whole 240 s recording (tools/make_reasm_golden.py --excerpt).
EXCERPT_SUS, EXCERPT_RECORDS = 520, 11


def test_recording_to_acars_end_to_end():
    """12 s of the 10.5k recording -> device demodulator -> device P-channel frame layer -> host reassembly == the signal units
    and ACARS records the reference's own demodulator + reassembly code produce (tests/golden/reasm_golden.json and
    reasm_su_streams.npz, made from the whole recording by tools/make_reasm_golden.py)."""
    import json
    import reasm_synth
    jb = _import()
    gold = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    pcm = load_excerpt("oqpsk_10500")
    with open(os.path.join(gold, "reasm_golden.json")) as fh:
        want = json.load(fh)["p_recording_10500"]["records"][:EXCERPT_RECORDS]
    want_sus = reasm_synth.unpack_stream(np.load(os.path.join(gold, "reasm_su_streams.npz"))["p_recording_10500"])[:EXCERPT_SUS]
    assert sum(1 for w in want if w["kind"] == 0 and not w["nonacars"]) == 6
    kw = dict(fb=10500, freq_center=5760, lockingbw=10500, fft_power=14, signalthreshold=0.65, afc=True)
    b = jb.DemodBatch("oqpsk", 2, **kw)
    pc = jb.PChannelBatch(2, 10500)
    rs = [jb.Reassembler(), jb.Reassembler()]
    sus = [[], []]
    chunk = 4800

    def drain():
        for c, (su, ok, _, _) in enumerate(pc.read_sus()):
            for k in range(len(ok)):
                if ok[k]:
                    sus[c].append(bytes(su[k, :10])); rs[c].push_su(su[k])

    for k, a in enumerate(range(0, len(pcm), chunk)):
        x = pcm[a:a + chunk]
        b.write(np.stack([x, x]))
        pc.process_softbits(b.read_softbits())
        if k % 5 == 4:
            drain()
    drain()
    for c in range(2):
        assert sus[c] == [e[1] for e in want_sus]                        # the CRC-valid signal units, byte for byte
        got = rs[c].pop_all()
        assert len(got) == len(want)
        for g, w in zip(got, want):
            assert g["kind"] == w["kind"] and g["aesid"] == w["aesid"] and g["text"] == bytes.fromhex(w["message"])
            assert g["reg"] == bytes.fromhex(w["reg"]) and g["label"] == bytes.fromhex(w["label"]) and g["bi"] == w["bi"]
        rs[c].close()
    b.close(); pc.close()


def test_error_behaviour():
    jb = _import()
    b = jb.DemodBatch("oqpsk", 2, fb=10500, freq_center=5760)
    b.write(np.zeros((2, 0), dtype=np.int16))                      # `if(!len)return 0;`
    pcm = load_excerpt("oqpsk_10500")[:48000 * 6]
    b.write(np.stack([pcm, pcm]))                                   # 6 s without draining: ring of 2 s overflows
    with pytest.raises(jb.JaeroError, match="overflow"):
        b.read_softbits()
    with pytest.raises(jb.JaeroError):
        jb.DemodBatch("oqpsk", 2, fb=10500, Fs=44100)              # unsupported rate: refuses, no fallback
    with pytest.raises(jb.JaeroError):
        jb.DemodBatch("msk", 0, fb=600)
    b.close()
