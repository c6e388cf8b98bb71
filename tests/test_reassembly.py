"""ISU/SSU reassembly + ACARS parsing (SURVEY.md section 8(f)4, host side; no GPU needed).

Golden records come from the reference's own code (JAERO/aerol.cpp:4-487 compiled verbatim, oracle/ref_reasm_driver.cpp)
run by tools/make_reasm_golden.py over (1) the CRC-valid P-channel signal units the reference demodulator produces from
the 240 s 10.5k recording, and (2) seeded synthetic streams (tests/reasm_synth.py); for further random streams the
reference's results are stored as digests (tests/ref_pins.py)."""
import hashlib
import json
import os

import numpy as np
import pytest

import jaero_b200
import reasm_synth
from ref_pins import digest, pinned

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden")


def _gold():
    with open(os.path.join(GOLD, "reasm_golden.json")) as fh:
        g = json.load(fh)
    z = np.load(os.path.join(GOLD, "reasm_su_streams.npz"))
    return g, {k: reasm_synth.unpack_stream(z[k]) for k in z.files}


def _run_product(stream):
    r = jaero_b200.Reassembler()
    rcs = []
    for e in stream:
        if e[0] == "su":
            rcs.append(r.push_su(e[1], e[2]))
        elif e[0] == "r":
            rcs.append(r.push_r(e[1], e[2]))
        elif e[0] == "reset":
            r.reset(); rcs.append(0)
        else:
            r.short_frame(); rcs.append(0)
    out = r.pop_all()
    st = r.stats()
    r.close()
    return rcs, out, st


def _same(got, want):
    """product record (dict with bytes) against a reference record (hex strings, see oracle/ref.py reasm_record)"""
    assert got["kind"] == want["kind"], (got, want)
    assert got["text"] == bytes.fromhex(want["message"]), (got, want)      # kind 1: the Errorsignal string (names the ISU)
    if want["kind"] == 0:
        for k in ("aesid", "gesid", "qno", "refno", "seqno", "nooct", "mode", "tak", "bi", "nonacars", "downlink", "valid", "hastext", "moretocome"):
            assert got[k] == want[k], (k, got, want)
        assert got["label"] == bytes.fromhex(want["label"])
        assert got["reg"] == bytes.fromhex(want["reg"])
        assert got["userdata_len"] == len(want["userdata"]) // 2


@pytest.mark.parametrize("name", ["p_recording_10500", "p_recording_600", "rt_recording_burst_oqpsk_10500", "rt_recording_burst_msk_1200_a", "rt_recording_burst_msk_1200_b",
                                  "p_synthetic", "t_synthetic", "r_synthetic", "garbage"])
def test_reassembly_matches_reference_golden(name):
    gold, streams = _gold()
    rcs, out, st = _run_product(streams[name])
    want = gold[name]
    assert rcs == want["return_codes"]
    assert len(out) == len(want["records"])
    for g, w in zip(out, want["records"]):
        _same(g, w)
    assert st["messages"] == sum(1 for w in want["records"] if w["kind"] == 0)
    assert st["errors"] == sum(1 for w in want["records"] if w["kind"] == 1)


def test_recording_yields_real_acars():
    """the recording's CRC-valid SUs reassemble into ACARS blocks with plausible registrations (sanity of the fixture)"""
    gold, streams = _gold()
    _, out, st = _run_product(streams["p_recording_10500"])
    acars = [o for o in out if o["kind"] == 0 and not o["nonacars"]]
    assert len(acars) >= 50
    assert all(len(o["reg"]) >= 5 and o["reg"].replace(b"-", b"").isalnum() for o in acars)
    assert st["isus"] >= len(out)


def test_t_packet_entry_point():
    """jaero_reasm_push_t_packet walks the SUs of a T packet the way AeroL::Decode does (JAERO/aerol.cpp:1480-1516)"""
    ud = reasm_synth.acars_userdata("G-ABCD", "H1", ord("D"), "HELLO FROM THE T CHANNEL")
    sus = reasm_synth.isu_to_sus(0x4ACA11, 0x90, 5, 2, ud)
    fill = bytes([0x01]) + bytes(11)
    info = bytes([0x4A, 0xCA, 0x11, 0x90, 0, 0]) + b"".join(s + b"\0\0" for s in sus[:3]) + fill
    info2 = bytes([0x4A, 0xCA, 0x11, 0x90, 0, 0]) + b"".join(s + b"\0\0" for s in sus[3:])
    r = jaero_b200.Reassembler()
    assert r.push_t_packet(info, 4) == 0
    rc = r.push_t_packet(info2, len(sus) - 3)
    assert rc & r.COMPLETE and rc & r.PARSED
    out = r.pop_all()
    assert len(out) == 1 and out[0]["text"] == b"HELLO FROM THE T CHANNEL" and out[0]["reg"] == b"G-ABCD" and out[0]["downlink"]
    r.close()


def test_pop_with_small_buffer():
    import ctypes
    ud = reasm_synth.acars_userdata("G-ABCD", "H1", ord("D"), "X" * 100)
    r = jaero_b200.Reassembler()
    for s in reasm_synth.isu_to_sus(0x4ACA11, 0x90, 5, 2, ud):
        r.push_su(s)
    L = jaero_b200.lib()
    rec = jaero_b200.AcarsRecord(); buf = ctypes.create_string_buffer(10)
    assert L.jaero_reasm_pending(r.h) == 1
    assert L.jaero_reasm_pop(r.h, ctypes.byref(rec), buf, 10) == -2 and rec.text_len == 100
    assert L.jaero_reasm_pending(r.h) == 1
    assert len(r.pop_all()[0]["text"]) == 100
    assert L.jaero_reasm_pop(r.h, ctypes.byref(rec), buf, 10) == -1
    r.close()


_FIELDS = ("aesid", "gesid", "qno", "refno", "seqno", "nooct", "mode", "tak", "bi", "nonacars", "downlink", "valid", "hastext", "moretocome")


def _canon_ref(w):
    """the parts of a reference record that _same compares, as JSON-able values"""
    if w["kind"] != 0:
        return [w["kind"], w["message"]]
    return [w["kind"], w["message"]] + [int(w[k]) for k in _FIELDS] + [w["label"], w["reg"], len(w["userdata"]) // 2]


def _canon_product(g):
    if g["kind"] != 0:
        return [g["kind"], g["text"].hex()]
    return [g["kind"], g["text"].hex()] + [int(g[k]) for k in _FIELDS] + [g["label"].hex(), g["reg"].hex(), g["userdata_len"]]


def _records_digest(canon):
    return [len(canon), hashlib.sha256(json.dumps(canon).encode()).hexdigest()]


@pytest.mark.parametrize("seed", [101, 102, 103])
def test_reassembly_matches_reference_live(seed):
    """fresh random streams against the reference's reassembly run on them (oracle/_ref/libjaero_ref_reasm.so), whose return
    codes and records are stored as digests in tests/golden/ref_pins.json"""
    stream = reasm_synth.p_stream(seed, burst=bool(seed & 1), n_msgs=50) + reasm_synth.r_stream(seed + 1, 40) + reasm_synth.garbage_stream(seed + 2, 1500)

    def run():
        from oracle import ref
        rr = ref.RefReasm()
        want_rc = []
        for e in stream:
            if e[0] == "su":
                want_rc.append(rr.push_su(e[1], e[2]))
            elif e[0] == "r":
                want_rc.append(rr.push_r(e[1], e[2]))
            elif e[0] == "reset":
                rr.reset(); want_rc.append(0)
            else:
                rr.short_frame(); want_rc.append(0)
        want = rr.pop_all(); rr.close()
        return [np.array(want_rc), _records_digest([_canon_ref(w) for w in want])]
    rcs, out, _ = _run_product(stream)
    want_rc, want = pinned("reasm/live_%d" % seed, run)
    assert digest(np.array(rcs)) == want_rc
    assert _records_digest([_canon_product(g) for g in out]) == want


@pytest.mark.parametrize("name", ["p_recording_10500", "p_recording_600", "rt_recording_burst_oqpsk_10500", "p_synthetic", "t_synthetic", "r_synthetic", "garbage"])
def test_restated_oracle_matches_reference_golden(name):
    """oracle/reasm_restated.py (the plain-Python restatement) is pinned by the verbatim reference build's golden records"""
    from oracle import reasm_restated
    gold, streams = _gold()
    o = reasm_restated.Reassembly()
    rcs = []
    for e in streams[name]:
        if e[0] == "su":
            rcs.append(o.push_su(e[1], e[2]))
        elif e[0] == "r":
            rcs.append(o.push_r(e[1], e[2]))
        elif e[0] == "reset":
            o.reset(); rcs.append(0)
        else:
            o.short_frame(); rcs.append(0)
    got = o.pop_all()
    want = gold[name]
    assert rcs == want["return_codes"]
    assert len(got) == len(want["records"])
    for g, w in zip(got, want["records"]):
        if w["kind"] == 1:
            assert g["kind"] == 1 and g["message"] == w["message"]
        else:
            assert g == {k: w[k] for k in g}, (g, w)


def test_reassembly_randomised_against_restated_oracle():
    """hypothesis-driven streams (structured messages with losses, duplicates, interleaving, raw garbage, resets): the product
    and the plain-Python restatement must agree record for record; runs everywhere (no oracle/_ref needed)"""
    from hypothesis import given, settings, strategies as st
    from oracle import reasm_restated

    su = st.one_of(
        st.builds(lambda b: ("su", bytes([0x71, 0, 0, b[0] & 3, b[1] & 1, b[2] & 0x11, b[3] & 3, b[4] & 0xF0]) + bytes(b[5:7]), bool(b[7] & 1)),
                  st.binary(min_size=8, max_size=8)),
        st.builds(lambda b: ("su", bytes([0xC0 | (b[0] & 3), b[1] & 0x11]) + bytes(b[2:10]), bool(b[0] & 4)), st.binary(min_size=10, max_size=10)),
        st.builds(lambda b: ("r", bytes([b[0], (b[1] & 0x11) | 0x08, 0, 0, b[2] & 1, b[3] & 1]) + bytes(b[4:15]), True), st.binary(min_size=15, max_size=15)),
        st.builds(lambda b: ("su", bytes(b), False), st.binary(min_size=10, max_size=10)),
        st.just(("reset",)), st.just(("short",)))
    msg = st.builds(lambda seed, burst: reasm_synth.p_stream(seed, burst=burst, n_msgs=3), st.integers(0, 10 ** 6), st.booleans())
    stream = st.lists(st.one_of(st.lists(su, max_size=40), msg), max_size=6).map(lambda parts: [e for p in parts for e in p])

    @settings(max_examples=60, deadline=None)
    @given(stream)
    def check(ev):
        o = reasm_restated.Reassembly()
        want_rc = []
        for e in ev:
            if e[0] == "su":
                want_rc.append(o.push_su(e[1], e[2]))
            elif e[0] == "r":
                want_rc.append(o.push_r(e[1], e[2]))
            elif e[0] == "reset":
                o.reset(); want_rc.append(0)
            else:
                o.short_frame(); want_rc.append(0)
        want = o.pop_all()
        rcs, out, _ = _run_product(ev)
        assert rcs == want_rc and len(out) == len(want)
        for g, w in zip(out, want):
            assert g["kind"] == w["kind"] and g["text"] == bytes.fromhex(w["message"])
            if w["kind"] == 0:
                for k in ("aesid", "gesid", "qno", "refno", "seqno", "nooct", "mode", "tak", "bi", "nonacars", "downlink", "hastext", "moretocome"):
                    assert g[k] == w[k], (k, g, w)
                assert g["label"] == bytes.fromhex(w["label"]) and g["reg"] == bytes.fromhex(w["reg"])

    check()
