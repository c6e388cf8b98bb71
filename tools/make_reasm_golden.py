"""Generate tests/golden/reasm_golden.json: the reference's own ISU/SSU reassembly + ACARS parse (oracle/_ref/
libjaero_ref_reasm.so = JAERO/aerol.cpp:4-487 compiled verbatim) run over
  (1) the CRC-valid P-channel signal units of the full 10.5k recording (tests/golden/pcm_full/oqpsk_10500.npy,
      demodulated by the verbatim reference demodulator, framed by the restated AeroL P-channel decoder);
  (2) the CRC-valid T/R packets of the burst recordings;
  (3) seeded synthetic SU streams that exercise multi-block ACARS, interleaved sequences, lost SSUs, parity errors,
      R-channel 1/2/3-SU sequences and the garbage cases.
The SU byte streams themselves are committed (tests/golden/reasm_su_streams.npz) so the tests need neither the
recordings nor the reference. Needs oracle/_ref and the full recordings (tools/make_fixtures.py); --excerpt needs only
oracle/_ref and prints how much of the recording's golden the committed 12 s excerpt covers."""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle import ref, restated  # noqa: E402
import reasm_synth  # noqa: E402  (tests/reasm_synth.py)


def recording_sus(name="oqpsk_10500", kind="oqpsk", kw=None, pcm=None):
    import multiprocessing as mp
    if pcm is None:
        pcm = np.load(os.path.join(ROOT, "tests", "golden", "pcm_full", name + ".npy"))
    kw = kw or dict(fb=10500, freq_center=5760, lockingbw=10500, fft_power=14, signalthreshold=0.65, afc=True)
    ctx = mp.get_context("spawn")
    with ctx.Pool(1) as pool:
        soft, state, cfe = pool.apply(ref.run_demod_job, ((kind, kw, pcm, 4800, None),))
    p = restated.OraclePChannel(kw["fb"])
    p.process(soft)
    su, ok, fr = p.take_sus()
    print("recording: %d SUs, %d CRC ok" % (len(ok), int(ok.sum())))
    return su[ok != 0][:, :10].copy()


def burst_recording_events(name, kind, kw):
    """R/T packets of a full-length burst recording (verbatim reference demodulator, restated R/T packet layer whose packets
    are CRC-16 verified) as reassembly events, in AeroL::Decode's order (JAERO/aerol.cpp:1357-1399, 1480-1516)."""
    import multiprocessing as mp
    pcm = np.load(os.path.join(ROOT, "tests", "golden", "pcm_full", name + ".npy"))
    ctx = mp.get_context("spawn")
    with ctx.Pool(1) as pool:
        soft, state, cfe = pool.apply(ref.run_demod_job, ((kind, kw, pcm, 4800, None),))
    rt = restated.OracleRTChannel(kw["fb"])
    rt.process(soft)
    ev = []
    for q in rt.packets():
        b = bytes(q["bytes"])
        if q["type"] == 1:
            ev.append(("r", b[:17], True))
        else:
            for k in range(q["nsus"]):
                ev.append(("su", b[6 + 12 * k:6 + 12 * k + 10], True))
    print(name, "packets", len(rt.packets()), "events", len(ev))
    return ev


def run_stream(stream):
    r = ref.RefReasm()
    rcs = []
    for e in stream:
        kind = e[0]
        if kind == "su":
            rcs.append(r.push_su(e[1], e[2]))
        elif kind == "r":
            rcs.append(r.push_r(e[1], e[2]))
        elif kind == "reset":
            r.reset(); rcs.append(0)
        elif kind == "short":
            r.short_frame(); rcs.append(0)
    out = r.pop_all()
    r.close()
    return rcs, out


def excerpt_prefix():
    """The committed 12 s excerpt through the same chain: its CRC-valid SUs and reassembled records must be a prefix of the
    whole recording's (tests/test_gpu_parity.py EXCERPT_SUS, EXCERPT_RECORDS)."""
    import json
    sus = recording_sus(pcm=np.load(os.path.join(ROOT, "tests", "golden", "oqpsk_10500_excerpt.npz"))["pcm"])
    full = reasm_synth.unpack_stream(np.load(os.path.join(ROOT, "tests", "golden", "reasm_su_streams.npz"))["p_recording_10500"])
    _, out = run_stream([("su", bytes(x), False) for x in sus])
    with open(os.path.join(ROOT, "tests", "golden", "reasm_golden.json")) as fh:
        gold = json.load(fh)["p_recording_10500"]["records"]
    assert [bytes(x) for x in sus] == [e[1] for e in full[:len(sus)]] and out == gold[:len(out)]
    print("EXCERPT_SUS, EXCERPT_RECORDS = %d, %d" % (len(sus), len(out)))


if __name__ == "__main__" and sys.argv[1:] == ["--excerpt"]:
    excerpt_prefix()
elif __name__ == "__main__":
    streams = {}
    rec = recording_sus()
    streams["p_recording_10500"] = [("su", bytes(x), False) for x in rec]
    rec600 = recording_sus("msk_600", "msk", dict(fb=600, freq_center=1000, lockingbw=900, fft_power=13, signalthreshold=0.5, afc=True))
    streams["p_recording_600"] = [("su", bytes(x), False) for x in rec600]      # BASELINE configs[0]: decoded ISUs of the 600 bps recording
    streams["rt_recording_burst_oqpsk_10500"] = burst_recording_events(
        "burst_oqpsk_10500", "burst_oqpsk", dict(fb=10500.0, freq_center=8000.0, lockingbw=10500.0, signalthreshold=0.6))
    for nm in ("burst_msk_1200_a", "burst_msk_1200_b"):
        streams["rt_recording_" + nm] = burst_recording_events(nm, "burst_msk", dict(fb=1200.0, freq_center=1000.0, lockingbw=1800.0, signalthreshold=0.6))
    for name, s in reasm_synth.synthetic_streams().items():
        streams[name] = s
    gold = {}
    arrays = {}
    for name, s in streams.items():
        rcs, out = run_stream(s)
        gold[name] = dict(return_codes=rcs, records=out)
        arrays[name] = reasm_synth.pack_stream(s)
        n_acars = sum(1 for o in out if o["kind"] == 0 and not o["nonacars"])
        print(name, "events", len(s), "records", len(out), "acars", n_acars, "errors", sum(1 for o in out if o["kind"] == 1))
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "reasm_su_streams.npz"), **arrays)
    with open(os.path.join(ROOT, "tests", "golden", "reasm_golden.json"), "w") as fh:
        json.dump(gold, fh, indent=0, sort_keys=True)
