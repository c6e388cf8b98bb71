"""TEST INFRASTRUCTURE ONLY. ctypes bindings for oracle/_build/libjaero_oracle.so — this repo's CPU
restatement of the reference's hot path (oracle/restated/*.cpp, oracle/correct_restated.c).
Only tests/, bench.py's cpu_baseline / --impl reference legs and __graft_entry__.smoke() may import this."""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "libjaero_oracle.so")
_lib = None
STATE_FIELDS = ["mixer2_freq", "mixer2_wtptr", "center_freq", "st_freq", "st_wtptr", "agc", "mse",
                "ebno", "marg", "cfe_est", "n_sig_true", "n_sig_false", "center_wtptr", "st_ref_wtptr"]


BURST_STATE_FIELDS = ["mixer2_freq", "mixer2_wtptr", "center_freq", "st_freq", "st_wtptr", "agc", "mse",
                      "ebno", "vol_gain", "rotator_freq", "n_sig_true", "n_sig_false", "cntr", "startstop"]


def available():
    return os.path.exists(_SO)


def lib():
    global _lib
    if _lib is None:
        L = ctypes.CDLL(_SO)
        vp, d, i, l = ctypes.c_void_p, ctypes.c_double, ctypes.c_int, ctypes.c_long
        L.jor_demod_new.restype = vp; L.jor_demod_new.argtypes = [i, d, d, d, d, i, d, i, i, i]
        L.jor_burst_msk_new.restype = vp; L.jor_burst_msk_new.argtypes = [d, d, d, d, d]
        L.jor_burst_oqpsk_new.restype = vp; L.jor_burst_oqpsk_new.argtypes = [d, d, d, d, d]
        L.jor_aux_take.restype = l; L.jor_aux_take.argtypes = [vp, i, vp, l]
        L.jor_write.argtypes = [vp, vp, l]; L.jor_set_dcd.argtypes = [vp, i]
        L.jor_soft_count.restype = l; L.jor_soft_count.argtypes = [vp]
        L.jor_soft_take.restype = l; L.jor_soft_take.argtypes = [vp, vp, l]
        L.jor_cfe_log_take.restype = l; L.jor_cfe_log_take.argtypes = [vp, vp, l]
        L.jor_state.argtypes = [vp, vp]; L.jor_free.argtypes = [vp]
        L.jor_rrc_design.argtypes = [d, i, d, d, vp, i]
        L.jor_trig_tables.argtypes = [vp, vp]; L.jor_qround.argtypes = [d]
        L.jor_fft.argtypes = [i, i, vp, vp]
        L.jor_jfastfir_rrc.argtypes = [d, i, d, d, i, vp, l]
        L.jor_cfe_new.restype = vp; L.jor_cfe_new.argtypes = [i, d, d, d]
        L.jor_cfe_process.restype = d; L.jor_cfe_process.argtypes = [vp, vp, vp, vp]
        L.jor_cfe_bigchange.argtypes = [vp]; L.jor_cfe_free.argtypes = [vp]
        L.jor_deinterleave.argtypes = [vp, i, vp]
        L.jor_viterbi_new.restype = vp; L.jor_viterbi_new.argtypes = [i]
        L.jor_viterbi_decode_continuous.argtypes = [vp, vp, i, vp]; L.jor_viterbi_free.argtypes = [vp]
        L.jor_conv_decode_soft.argtypes = [vp, i, vp]; L.jor_conv_encode.argtypes = [vp, i, vp]
        L.jor_pchan_new.restype = vp; L.jor_pchan_new.argtypes = [i]
        L.jor_pchan_process.argtypes = [vp, vp, i]; L.jor_pchan_update_dcd.argtypes = [vp]
        L.jor_pchan_dcd.argtypes = [vp]
        L.jor_pchan_lost_signal.argtypes = [vp]; L.jor_wire_pchan.argtypes = [vp, vp]
        L.jor_pchan_su_count.restype = l; L.jor_pchan_su_count.argtypes = [vp]
        L.jor_pchan_su_take.restype = l; L.jor_pchan_su_take.argtypes = [vp, vp, vp, vp, l]
        L.jor_pchan_free.argtypes = [vp]
        L.jor_crc16.restype = ctypes.c_uint16; L.jor_crc16.argtypes = [vp, i]
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


class OracleDemod:
    def __init__(self, kind, fb, Fs=48000.0, freq_center=8000.0, lockingbw=10500.0, fft_power=14,
                 signalthreshold=0.65, afc=False, sql=False, cpureduce=False):
        self.kind = kind
        if kind == "burst_msk":
            self.h = lib().jor_burst_msk_new(fb, Fs, freq_center, lockingbw, signalthreshold)
        elif kind == "burst_oqpsk":
            self.h = lib().jor_burst_oqpsk_new(fb, Fs, freq_center, lockingbw, signalthreshold)
        else:
            self.h = lib().jor_demod_new(0 if kind == "oqpsk" else 1, fb, Fs, freq_center, lockingbw, fft_power,
                                         signalthreshold, int(afc), int(sql), int(cpureduce))

    def write(self, pcm):
        pcm = np.ascontiguousarray(pcm, dtype=np.int16)
        lib().jor_write(self.h, _p(pcm), len(pcm))

    def set_dcd(self, dcd):
        lib().jor_set_dcd(self.h, int(dcd))

    def take_soft(self):
        n = lib().jor_soft_count(self.h)
        out = np.zeros(n, dtype=np.int16)
        if n:
            lib().jor_soft_take(self.h, _p(out), n)
        return out

    def take_cfe_log(self):
        out = np.zeros(1 << 16, dtype=np.float64)
        n = lib().jor_cfe_log_take(self.h, _p(out), len(out))
        return out[:n].copy()

    def take_aux(self, which):
        out = np.zeros(1 << 14, dtype=np.float64)
        n = lib().jor_aux_take(self.h, which, _p(out), len(out))
        return out[:n].copy()

    def state(self):
        o = np.zeros(16, dtype=np.float64)
        n = lib().jor_state(self.h, _p(o))
        fields = BURST_STATE_FIELDS if self.kind.startswith("burst") else STATE_FIELDS
        return dict(zip(fields, o[:n]))

    def close(self):
        if self.h:
            lib().jor_free(self.h); self.h = None


class OracleViterbi:
    def __init__(self, paddinglength=24):
        self.h = lib().jor_viterbi_new(paddinglength)

    def decode_continuous(self, soft):
        soft = np.ascontiguousarray(soft, dtype=np.uint8)
        out = np.zeros(len(soft), dtype=np.int32)
        n = lib().jor_viterbi_decode_continuous(self.h, _p(soft), len(soft), _p(out))
        return out[:n].copy()

    def close(self):
        if self.h:
            lib().jor_viterbi_free(self.h); self.h = None


def conv_encode(msg_bytes):
    msg = np.ascontiguousarray(msg_bytes, dtype=np.uint8)
    enc = np.zeros(2 * (len(msg) + 2) + 8, dtype=np.uint8)
    nbits = lib().jor_conv_encode(_p(msg), len(msg), _p(enc))
    return np.unpackbits(enc)[:nbits]


def conv_decode_soft(soft):
    soft = np.ascontiguousarray(soft, dtype=np.uint8)
    msg = np.zeros(len(soft) // 16 + 8, dtype=np.uint8)
    nbytes = lib().jor_conv_decode_soft(_p(soft), len(soft), _p(msg))
    return np.unpackbits(msg[:nbytes])


def deinterleave(block, cols):
    block = np.ascontiguousarray(block, dtype=np.int32)
    out = np.zeros(64 * cols, dtype=np.uint8)
    lib().jor_deinterleave(_p(block), cols, _p(out))
    return out


class OraclePChannel:
    """Restated AeroL::Decode (continuous P-channel): soft bits -> signal units + CRC flags + DCD."""

    def __init__(self, fb):
        self.h = lib().jor_pchan_new(int(fb))

    def process(self, soft):
        soft = np.ascontiguousarray(soft, dtype=np.int16)
        lib().jor_pchan_process(self.h, _p(soft), len(soft))

    def update_dcd(self):
        lib().jor_pchan_update_dcd(self.h)

    def lost_signal(self):
        """AeroL::LostSignal (aerol.h:925-931)"""
        lib().jor_pchan_lost_signal(self.h)

    def wire(self, demod):
        """Connect a continuous OracleDemod to this AeroL as JAERO/mainwindow.cpp does (direct connections): soft-bit vectors are
        decoded inside write(), DCD and LostSignal feed back at once. take_soft() on the demodulator still returns what was emitted."""
        lib().jor_wire_pchan(demod.h, self.h)

    @property
    def dcd(self):
        return bool(lib().jor_pchan_dcd(self.h))

    def take_sus(self):
        n = lib().jor_pchan_su_count(self.h)
        b = np.zeros((n, 12), dtype=np.uint8); ok = np.zeros(n, dtype=np.int32); fr = np.zeros(n, dtype=np.int64)
        if n:
            lib().jor_pchan_su_take(self.h, _p(b), _p(ok), _p(fr), n)
        return b, ok, fr

    def close(self):
        if self.h:
            lib().jor_pchan_free(self.h); self.h = None


class OracleRTChannel:
    """Restated burst branch of AeroL::Decode + RTChannelDeleaveFECScram: soft bits (with -1 markers) -> R / T packets."""

    def __init__(self, fb):
        L = lib()
        L.jor_rt_new.restype = ctypes.c_void_p; L.jor_rt_new.argtypes = [ctypes.c_int]
        L.jor_rt_process.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int]
        L.jor_rt_update_dcd.argtypes = [ctypes.c_void_p]
        L.jor_rt_packet_count.restype = ctypes.c_long; L.jor_rt_packet_count.argtypes = [ctypes.c_void_p]
        L.jor_rt_trials.restype = ctypes.c_long; L.jor_rt_trials.argtypes = [ctypes.c_void_p]
        L.jor_rt_packet.argtypes = [ctypes.c_void_p, ctypes.c_long, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int]
        L.jor_rt_free.argtypes = [ctypes.c_void_p]
        self.h = L.jor_rt_new(int(fb))

    def process(self, soft, vector_semantics=False):
        soft = np.ascontiguousarray(soft, dtype=np.int16)
        lib().jor_rt_process(self.h, _p(soft), len(soft), int(vector_semantics))

    def update_dcd(self):
        lib().jor_rt_update_dcd(self.h)

    @property
    def trials(self):
        return lib().jor_rt_trials(self.h)

    def packets(self):
        out = []
        for k in range(lib().jor_rt_packet_count(self.h)):
            t = ctypes.c_int(); ns = ctypes.c_int(); bi = ctypes.c_long(); buf = np.zeros(1024, dtype=np.uint8)
            n = lib().jor_rt_packet(self.h, k, ctypes.byref(t), ctypes.byref(ns), ctypes.byref(bi), _p(buf), 1024)
            out.append(dict(type=t.value, nsus=ns.value, bit_index=bi.value, bytes=buf[:n].copy()))
        return out

    def close(self):
        if self.h:
            lib().jor_rt_free(self.h); self.h = None


class OracleCChannel:
    """Restated AeroL::DecodeC (8400 bps C-channel): soft bits -> per frame 3 sub-band signal units (+CRC) and 25 x 12 voice bytes."""

    def __init__(self):
        L = lib()
        L.jor_cchan_new.restype = ctypes.c_void_p
        L.jor_cchan_process.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int]
        L.jor_cchan_update_dcd.argtypes = [ctypes.c_void_p]
        L.jor_cchan_dcd.argtypes = [ctypes.c_void_p]
        L.jor_cchan_frame_count.restype = ctypes.c_long; L.jor_cchan_frame_count.argtypes = [ctypes.c_void_p]
        L.jor_cchan_take.restype = ctypes.c_long; L.jor_cchan_take.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_long]
        L.jor_cchan_free.argtypes = [ctypes.c_void_p]
        self.h = L.jor_cchan_new()

    def process(self, soft):
        soft = np.ascontiguousarray(soft, dtype=np.int16)
        lib().jor_cchan_process(self.h, _p(soft), len(soft))

    def update_dcd(self):
        lib().jor_cchan_update_dcd(self.h)

    @property
    def dcd(self):
        return bool(lib().jor_cchan_dcd(self.h))

    def take_frames(self):
        n = lib().jor_cchan_frame_count(self.h)
        su = np.zeros((n, 3, 12), dtype=np.uint8); ok = np.zeros((n, 3), dtype=np.int32); voice = np.zeros((n, 300), dtype=np.uint8)
        if n:
            lib().jor_cchan_take(self.h, _p(su), _p(ok), _p(voice), n)
        return su, ok, voice

    def close(self):
        if self.h:
            lib().jor_cchan_free(self.h); self.h = None


def run_demod_job(args):
    """(kind, kw, pcm, chunk) -> (soft, state, aux0): one restated demodulator over one stream. Module-level so that tests can
    farm channels out to a multiprocessing pool."""
    kind, kw, pcm, chunk = args
    d = OracleDemod(kind, **kw)
    for a in range(0, len(pcm), chunk):
        d.write(pcm[a:a + chunk])
    soft, st = d.take_soft(), d.state()
    aux = d.take_aux(0) if kind.startswith("burst") else np.zeros(0)
    d.close()
    return soft, st, aux
