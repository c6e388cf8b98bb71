"""jaero_b200 — B200-native (sm_100a) batched implementation of JAERO's demodulator + Viterbi hot path.

This module is a thin ctypes loader over the C ABI in include/jaero_b200.h (libjaero_b200.so, built
in-tree by jaero_b200/build.py). There is no CPU fallback: constructing a batch without the CUDA
library or without a GPU raises.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("JAERO_B200_LIB", os.path.join(_HERE, "libjaero_b200.so"))   # override: kernel A/B experiments
KIND_OQPSK, KIND_MSK = 0, 1
_lib = None


class JaeroError(RuntimeError):
    pass


class Settings(ctypes.Structure):
    """Mirror of jaero_settings == the reference's Settings structs (oqpskdemodulator.h:20-39, mskdemodulator.h:24-45)."""
    _fields_ = [("kind", ctypes.c_int), ("coarsefreqest_fft_power", ctypes.c_int), ("freq_center", ctypes.c_double),
                ("lockingbw", ctypes.c_double), ("fb", ctypes.c_double), ("Fs", ctypes.c_double),
                ("signalthreshold", ctypes.c_double), ("afc", ctypes.c_int), ("sql", ctypes.c_int),
                ("cpu_reduce", ctypes.c_int), ("report_ebno", ctypes.c_int)]


class Status(ctypes.Structure):
    _fields_ = [(n, ctypes.c_double) for n in
                ("mixer2_freq", "mixer2_wtptr", "center_freq", "st_freq", "st_wtptr", "agc", "mse", "ebno", "marg",
                 "cfe_est", "n_sig_true", "n_sig_false", "center_wtptr", "st_ref_wtptr")] + \
               [("samples", ctypes.c_int64), ("softbits", ctypes.c_int64), ("dcd", ctypes.c_int32), ("reserved", ctypes.c_int32),
                ("peak_volume", ctypes.c_double), ("scatter", ctypes.c_double * 4)]


class AcarsRecord(ctypes.Structure):
    """jaero_acars_record (include/jaero_b200.h)."""
    _fields_ = [("kind", ctypes.c_int32), ("aes_id", ctypes.c_uint32),
                ("ges_id", ctypes.c_uint8), ("qno", ctypes.c_uint8), ("refno", ctypes.c_uint8), ("seqno", ctypes.c_uint8),
                ("last_octets", ctypes.c_uint8), ("mode", ctypes.c_uint8), ("tak", ctypes.c_uint8), ("block_id", ctypes.c_uint8),
                ("label", ctypes.c_uint8 * 2), ("label_len", ctypes.c_uint8), ("reg", ctypes.c_uint8 * 7), ("reg_len", ctypes.c_uint8),
                ("flags", ctypes.c_uint8), ("userdata_len", ctypes.c_uint32), ("text_len", ctypes.c_uint32)]


class ChanSettings(ctypes.Structure):
    """jaero_chan_settings (include/jaero_b200.h)."""
    _fields_ = [("iq_format", ctypes.c_int), ("reserved", ctypes.c_int), ("input_rate", ctypes.c_double),
                ("output_rate", ctypes.c_double), ("audio_hz", ctypes.c_double), ("passband_hz", ctypes.c_double),
                ("gain", ctypes.c_double)]


IQ_FORMATS = {"cs16": 0, "cu8": 1}


EXPORTS = ["jaero_last_error", "jaero_device_count", "jaero_batch_create", "jaero_batch_destroy", "jaero_batch_channels",
           "jaero_batch_write", "jaero_batch_write_device", "jaero_batch_sync", "jaero_batch_read_softbits",
           "jaero_batch_softbits_device", "jaero_batch_reset_softbits", "jaero_batch_set_dcd",
           "jaero_batch_set_center_freq", "jaero_batch_set_afc", "jaero_batch_set_sql", "jaero_batch_set_cpu_reduce", "jaero_batch_regroup",
           "jaero_burst_set_afc", "jaero_burst_set_sql", "jaero_batch_get_status", "jaero_batch_get_status_all",
           "jaero_batch_launch_count", "jaero_batch_set_stream", "jaero_batch_set_profiling",
           "jaero_batch_get_profile", "jaero_viterbi_create", "jaero_viterbi_destroy",
           "jaero_viterbi_decode_continuous", "jaero_viterbi_decode_continuous_device", "jaero_viterbi_decode_block",
           "jaero_viterbi_reset", "jaero_viterbi_sync", "jaero_viterbi_launch_count",
           "jaero_pchannel_create", "jaero_pchannel_destroy", "jaero_pchannel_process_batch",
           "jaero_pchannel_process_softbits", "jaero_pchannel_tick", "jaero_pchannel_read_sus",
           "jaero_pchannel_discard_sus", "jaero_pchannel_get_stats", "jaero_pchannel_launch_count", "jaero_pchannel_su_capacity",
           "jaero_pchannel_lost_signal", "jaero_pchannel_write_batch", "jaero_cchannel_lost_signal", "jaero_cchannel_write_batch", "jaero_batch_wire_signal_status",
           "jaero_burst_msk_create", "jaero_burst_oqpsk_create", "jaero_burst_destroy", "jaero_burst_write", "jaero_burst_write_device",
           "jaero_burst_read_softbits", "jaero_burst_set_dcd", "jaero_burst_get_status_all", "jaero_burst_sync",
           "jaero_burst_launch_count",
           "jaero_rt_create", "jaero_rt_destroy", "jaero_rt_process_softbits", "jaero_rt_process_burst", "jaero_rt_tick",
           "jaero_rt_read_packets", "jaero_rt_get_stats", "jaero_rt_launch_count", "jaero_rt_set_vector_mode",
           "jaero_cchannel_create", "jaero_cchannel_destroy", "jaero_cchannel_process_batch", "jaero_cchannel_process_softbits",
           "jaero_cchannel_tick", "jaero_cchannel_read_frames", "jaero_cchannel_get_stats", "jaero_cchannel_launch_count",
           "jaero_ingest_create", "jaero_ingest_destroy", "jaero_ingest_message", "jaero_ingest_available", "jaero_ingest_flush",
           "jaero_reasm_create", "jaero_reasm_destroy", "jaero_reasm_reset", "jaero_reasm_short_frame", "jaero_reasm_push_su",
           "jaero_reasm_push_r", "jaero_reasm_push_t_packet", "jaero_reasm_pending", "jaero_reasm_pop", "jaero_reasm_get_stats",
           "jaero_chan_taps", "jaero_chan_create", "jaero_chan_destroy", "jaero_chan_write", "jaero_chan_write_device",
           "jaero_chan_output_device", "jaero_chan_read", "jaero_chan_set_stream", "jaero_chan_sync", "jaero_chan_launch_count",
           "jaero_chan_ratio"]


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise JaeroError("libjaero_b200.so is not built (run `python -m jaero_b200.build`); there is no CPU fallback")
        L = ctypes.CDLL(LIB_PATH)
        vp, i, d, sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_double, ctypes.c_size_t
        L.jaero_last_error.restype = ctypes.c_char_p
        L.jaero_batch_create.argtypes = [ctypes.POINTER(Settings), i, vp, i, ctypes.POINTER(vp)]
        L.jaero_batch_destroy.argtypes = [vp]; L.jaero_batch_destroy.restype = None
        L.jaero_batch_channels.argtypes = [vp]
        L.jaero_batch_write.argtypes = [vp, vp, sz, sz]
        L.jaero_batch_write_device.argtypes = [vp, vp, sz, sz]
        L.jaero_batch_sync.argtypes = [vp]
        L.jaero_batch_read_softbits.argtypes = [vp, vp, sz, vp]
        L.jaero_batch_softbits_device.argtypes = [vp, ctypes.POINTER(vp), ctypes.POINTER(vp), ctypes.POINTER(sz)]
        L.jaero_batch_reset_softbits.argtypes = [vp]
        L.jaero_batch_set_dcd.argtypes = [vp, i, i]
        L.jaero_batch_set_center_freq.argtypes = [vp, i, d]
        L.jaero_batch_set_afc.argtypes = [vp, i]; L.jaero_batch_set_sql.argtypes = [vp, i]; L.jaero_batch_set_cpu_reduce.argtypes = [vp, i]
        L.jaero_burst_set_afc.argtypes = [vp, i]; L.jaero_burst_set_sql.argtypes = [vp, i]
        L.jaero_batch_get_status.argtypes = [vp, i, ctypes.POINTER(Status)]
        L.jaero_batch_get_status_all.argtypes = [vp, vp]
        L.jaero_batch_launch_count.argtypes = [vp]; L.jaero_batch_launch_count.restype = ctypes.c_int64
        L.jaero_batch_set_stream.argtypes = [vp, vp]
        L.jaero_batch_set_profiling.argtypes = [vp, i]
        L.jaero_batch_get_profile.argtypes = [vp, vp]
        L.jaero_viterbi_create.argtypes = [i, i, i, ctypes.POINTER(vp)]
        L.jaero_viterbi_destroy.argtypes = [vp]; L.jaero_viterbi_destroy.restype = None
        L.jaero_viterbi_decode_continuous.argtypes = [vp, vp, sz, i, vp, vp]
        L.jaero_viterbi_decode_continuous_device.argtypes = [vp, vp, sz, i, vp, vp]
        L.jaero_viterbi_decode_block.argtypes = [vp, vp, sz, vp]
        L.jaero_viterbi_reset.argtypes = [vp]; L.jaero_viterbi_sync.argtypes = [vp]
        L.jaero_viterbi_launch_count.argtypes = [vp]; L.jaero_viterbi_launch_count.restype = ctypes.c_int64
        L.jaero_pchannel_create.argtypes = [i, d, i, ctypes.POINTER(vp)]
        L.jaero_pchannel_destroy.argtypes = [vp]; L.jaero_pchannel_destroy.restype = None
        L.jaero_pchannel_process_batch.argtypes = [vp, vp]
        L.jaero_pchannel_process_softbits.argtypes = [vp, vp, sz, vp]
        L.jaero_pchannel_tick.argtypes = [vp, vp]
        L.jaero_pchannel_read_sus.argtypes = [vp, vp, sz, vp]
        L.jaero_pchannel_discard_sus.argtypes = [vp]
        L.jaero_pchannel_get_stats.argtypes = [vp, vp, vp, vp]
        L.jaero_pchannel_launch_count.argtypes = [vp]; L.jaero_pchannel_launch_count.restype = ctypes.c_int64
        L.jaero_pchannel_su_capacity.argtypes = [vp]
        L.jaero_pchannel_lost_signal.argtypes = [vp, vp, i]; L.jaero_cchannel_lost_signal.argtypes = [vp, vp, i]
        L.jaero_pchannel_write_batch.argtypes = [vp, vp, vp, sz, sz]; L.jaero_cchannel_write_batch.argtypes = [vp, vp, vp, sz, sz]
        L.jaero_batch_wire_signal_status.argtypes = [vp, i]
        L.jaero_batch_regroup.argtypes = [vp, vp]
        L.jaero_burst_msk_create.argtypes = [ctypes.POINTER(Settings), i, i, ctypes.POINTER(vp)]
        L.jaero_burst_oqpsk_create.argtypes = [ctypes.POINTER(Settings), i, i, ctypes.POINTER(vp)]
        L.jaero_burst_destroy.argtypes = [vp]; L.jaero_burst_destroy.restype = None
        L.jaero_burst_write.argtypes = [vp, vp, sz, sz]; L.jaero_burst_write_device.argtypes = [vp, vp, sz, sz]
        L.jaero_burst_read_softbits.argtypes = [vp, vp, sz, vp]
        L.jaero_burst_set_dcd.argtypes = [vp, i, i]
        L.jaero_burst_get_status_all.argtypes = [vp, vp]
        L.jaero_burst_sync.argtypes = [vp]
        L.jaero_burst_launch_count.argtypes = [vp]; L.jaero_burst_launch_count.restype = ctypes.c_int64
        L.jaero_rt_create.argtypes = [ctypes.c_double, i, i, ctypes.POINTER(vp)]
        L.jaero_rt_destroy.argtypes = [vp]; L.jaero_rt_destroy.restype = None
        L.jaero_rt_process_softbits.argtypes = [vp, vp, sz, vp]
        L.jaero_rt_process_burst.argtypes = [vp, vp]
        L.jaero_rt_tick.argtypes = [vp]; L.jaero_rt_set_vector_mode.argtypes = [vp, i]
        L.jaero_rt_read_packets.argtypes = [vp, vp, i, vp]
        L.jaero_rt_get_stats.argtypes = [vp, vp, vp, vp]
        L.jaero_rt_launch_count.argtypes = [vp]; L.jaero_rt_launch_count.restype = ctypes.c_int64
        L.jaero_cchannel_create.argtypes = [i, i, ctypes.POINTER(vp)]
        L.jaero_cchannel_destroy.argtypes = [vp]; L.jaero_cchannel_destroy.restype = None
        L.jaero_cchannel_process_batch.argtypes = [vp, vp]
        L.jaero_cchannel_process_softbits.argtypes = [vp, vp, sz, vp]
        L.jaero_cchannel_tick.argtypes = [vp, vp]
        L.jaero_cchannel_read_frames.argtypes = [vp, vp, i, vp]
        L.jaero_cchannel_get_stats.argtypes = [vp, vp, vp, vp]
        L.jaero_cchannel_launch_count.argtypes = [vp]; L.jaero_cchannel_launch_count.restype = ctypes.c_int64
        L.jaero_ingest_create.argtypes = [i, ctypes.POINTER(ctypes.c_char_p), ctypes.c_uint32, sz, ctypes.POINTER(vp)]
        L.jaero_ingest_destroy.argtypes = [vp]; L.jaero_ingest_destroy.restype = None
        L.jaero_ingest_message.argtypes = [vp, ctypes.c_char_p, sz, ctypes.c_char_p, sz, vp, sz]
        L.jaero_ingest_available.argtypes = [vp]; L.jaero_ingest_available.restype = sz
        L.jaero_ingest_flush.argtypes = [vp, vp, sz]
        L.jaero_reasm_create.argtypes = [ctypes.POINTER(vp)]
        L.jaero_reasm_destroy.argtypes = [vp]; L.jaero_reasm_destroy.restype = None
        L.jaero_reasm_reset.argtypes = [vp]; L.jaero_reasm_short_frame.argtypes = [vp]
        L.jaero_reasm_push_su.argtypes = [vp, ctypes.c_char_p, i]
        L.jaero_reasm_push_r.argtypes = [vp, ctypes.c_char_p, i]
        L.jaero_reasm_push_t_packet.argtypes = [vp, ctypes.c_char_p, i]
        L.jaero_reasm_pending.argtypes = [vp]
        L.jaero_reasm_pop.argtypes = [vp, ctypes.POINTER(AcarsRecord), vp, sz]; L.jaero_reasm_pop.restype = ctypes.c_long
        L.jaero_reasm_get_stats.argtypes = [vp, vp, vp, vp, vp]
        L.jaero_chan_taps.argtypes = [ctypes.POINTER(ChanSettings), vp, i]
        L.jaero_chan_ratio.argtypes = [ctypes.POINTER(ChanSettings), ctypes.POINTER(i), ctypes.POINTER(i)]
        L.jaero_chan_create.argtypes = [ctypes.POINTER(ChanSettings), i, vp, i, ctypes.POINTER(vp)]
        L.jaero_chan_destroy.argtypes = [vp]; L.jaero_chan_destroy.restype = None
        L.jaero_chan_write.argtypes = [vp, vp, sz]; L.jaero_chan_write_device.argtypes = [vp, vp, sz]
        L.jaero_chan_output_device.argtypes = [vp, ctypes.POINTER(vp), ctypes.POINTER(sz), ctypes.POINTER(sz)]
        L.jaero_chan_read.argtypes = [vp, vp, sz, ctypes.POINTER(sz)]
        L.jaero_chan_set_stream.argtypes = [vp, vp]; L.jaero_chan_sync.argtypes = [vp]
        L.jaero_chan_launch_count.argtypes = [vp]; L.jaero_chan_launch_count.restype = ctypes.c_int64
        _lib = L
    return _lib


def _check(rc):
    if rc != 0:
        raise JaeroError("jaero_b200 error %d: %s" % (rc, lib().jaero_last_error().decode()))


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


class DemodBatch:
    """n_channels independent continuous demodulators on one GPU (kind 'oqpsk' or 'msk').

    write() == the reference's writeData() for every channel; read_softbits() returns what the
    reference would have emitted through processDemodulatedSoftBits since the previous read."""

    def __init__(self, kind, n_channels, fb, Fs=48000.0, freq_center=8000.0, lockingbw=10500.0, fft_power=None,
                 signalthreshold=None, afc=False, sql=False, cpu_reduce=False, report_ebno=True, device=0):
        k = KIND_OQPSK if kind == "oqpsk" else KIND_MSK
        if fft_power is None:
            fft_power = 14 if k == KIND_OQPSK else 13
        if signalthreshold is None:
            signalthreshold = 0.65 if k == KIND_OQPSK else 0.5
        if n_channels <= 0:
            raise JaeroError("n_channels must be positive")
        fc = np.ascontiguousarray(np.broadcast_to(np.asarray(freq_center, dtype=np.float64), (n_channels,)))
        s = Settings(k, fft_power, float(fc[0]), lockingbw, fb, Fs, signalthreshold, int(afc), int(sql), int(cpu_reduce), int(report_ebno))
        self.h = ctypes.c_void_p()
        self.n = n_channels
        self.kind = kind
        self.soft_cap = max(4096, int(2 * fb) + 64)
        _check(lib().jaero_batch_create(ctypes.byref(s), n_channels, _p(fc), device, ctypes.byref(self.h)))

    def write(self, pcm):
        """pcm: int16 array [n_channels, n_samples] (host)."""
        pcm = np.asarray(pcm)
        assert pcm.dtype == np.int16 and pcm.ndim == 2 and pcm.shape[0] == self.n
        if not pcm.flags.c_contiguous:
            pcm = np.ascontiguousarray(pcm)
        _check(lib().jaero_batch_write(self.h, _p(pcm), pcm.shape[1], pcm.strides[0] // 2 if pcm.shape[0] > 1 else pcm.shape[1]))

    def write_device(self, dev_ptr, n_samples, stride):
        _check(lib().jaero_batch_write_device(self.h, ctypes.c_void_p(dev_ptr), n_samples, stride))

    def sync(self):
        _check(lib().jaero_batch_sync(self.h))

    def set_afc(self, state):
        """setAFC / setSQL / setCPUReduce of the reference classes, every channel, from the next write on"""
        _check(lib().jaero_batch_set_afc(self.h, int(bool(state))))

    def set_sql(self, state):
        _check(lib().jaero_batch_set_sql(self.h, int(bool(state))))

    def set_cpu_reduce(self, state):
        _check(lib().jaero_batch_set_cpu_reduce(self.h, int(bool(state))))

    def regroup(self, slot_of=None):
        """seat the channels by symbol-timing phase now (slot_of None) or as the given permutation; never changes results"""
        if slot_of is None:
            _check(lib().jaero_batch_regroup(self.h, None))
        else:
            a = np.ascontiguousarray(slot_of, dtype=np.int32)
            assert len(a) == self.n
            _check(lib().jaero_batch_regroup(self.h, _p(a)))

    def wire_signal_status(self, on=True):
        """connect(demodulator, SignalStatus, aerol, SignalStatusSlot) (mainwindow.cpp:432,508)"""
        _check(lib().jaero_batch_wire_signal_status(self.h, int(bool(on))))

    def read_softbits(self):
        out = np.zeros((self.n, self.soft_cap), dtype=np.int16)
        counts = np.zeros(self.n, dtype=np.int32)
        _check(lib().jaero_batch_read_softbits(self.h, _p(out), self.soft_cap, _p(counts)))
        return [out[c, :counts[c]].copy() for c in range(self.n)]

    def reset_softbits(self):
        _check(lib().jaero_batch_reset_softbits(self.h))

    def softbits_device(self):
        a, b, c = ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_size_t()
        _check(lib().jaero_batch_softbits_device(self.h, ctypes.byref(a), ctypes.byref(b), ctypes.byref(c)))
        return a.value, b.value, c.value

    def set_dcd(self, dcd, channel=-1):
        _check(lib().jaero_batch_set_dcd(self.h, channel, int(dcd)))

    def set_center_freq(self, hz, channel=-1):
        _check(lib().jaero_batch_set_center_freq(self.h, channel, float(hz)))

    def status(self):
        arr = (Status * self.n)()
        _check(lib().jaero_batch_get_status_all(self.h, ctypes.cast(arr, ctypes.c_void_p)))
        return [{f[0]: getattr(arr[c], f[0]) for f in Status._fields_} for c in range(self.n)]

    def set_stream(self, cuda_stream):
        _check(lib().jaero_batch_set_stream(self.h, ctypes.c_void_p(cuda_stream)))

    def set_profiling(self, on):
        _check(lib().jaero_batch_set_profiling(self.h, int(on)))

    def get_profile(self):
        o = np.zeros(5, dtype=np.float64)
        _check(lib().jaero_batch_get_profile(self.h, _p(o)))
        return dict(segment_ms=o[0], segment_launches=int(o[1]), cfe_ms=o[2], cfe_runs=int(o[3]), samples=int(o[4]))

    @property
    def launches(self):
        return lib().jaero_batch_launch_count(self.h)

    def close(self):
        if self.h:
            lib().jaero_batch_destroy(self.h); self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class ViterbiBatch:
    """Batched JConvolutionalCodec (K=7, r=1/2, polys 109/79): Decode_Continuous / Decode_soft."""

    def __init__(self, n_channels, paddinglength=24, device=0):
        self.h = ctypes.c_void_p()
        self.n = n_channels
        _check(lib().jaero_viterbi_create(n_channels, paddinglength, device, ctypes.byref(self.h)))

    def decode_continuous(self, soft, interleaver_cols=0):
        soft = np.ascontiguousarray(soft, dtype=np.uint8)
        assert soft.ndim == 2 and soft.shape[0] == self.n
        out = np.zeros((self.n, soft.shape[1] // 2), dtype=np.uint8)
        valid = np.zeros(self.n, dtype=np.int32)
        _check(lib().jaero_viterbi_decode_continuous(self.h, _p(soft), soft.shape[1], interleaver_cols, _p(out), _p(valid)))
        self.last_valid = valid
        return out

    def decode_continuous_device(self, d_soft, n_soft, interleaver_cols, d_bits, d_valid=None):
        _check(lib().jaero_viterbi_decode_continuous_device(self.h, ctypes.c_void_p(d_soft), n_soft, interleaver_cols,
                                                            ctypes.c_void_p(d_bits), ctypes.c_void_p(d_valid)))

    def decode_block(self, soft):
        soft = np.ascontiguousarray(soft, dtype=np.uint8)
        out = np.zeros((self.n, soft.shape[1] // 2), dtype=np.uint8)
        _check(lib().jaero_viterbi_decode_block(self.h, _p(soft), soft.shape[1], _p(out)))
        return out

    def reset(self):
        _check(lib().jaero_viterbi_reset(self.h))

    def sync(self):
        _check(lib().jaero_viterbi_sync(self.h))

    @property
    def launches(self):
        return lib().jaero_viterbi_launch_count(self.h)

    def close(self):
        if self.h:
            lib().jaero_viterbi_destroy(self.h); self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class PChannelBatch:
    """Batched AeroL P-channel frame layer (600/1200/10500 bps, continuous): soft bits -> CRC-checked SUs + DCD."""

    def __init__(self, n_channels, fb, device=0):
        self.h = ctypes.c_void_p()
        self.n = n_channels
        _check(lib().jaero_pchannel_create(n_channels, float(fb), device, ctypes.byref(self.h)))
        self.su_cap = int(lib().jaero_pchannel_su_capacity(self.h))

    def process_batch(self, batch):
        _check(lib().jaero_pchannel_process_batch(self.h, batch.h))

    def process_softbits(self, soft_list):
        cap = max(1, max(len(s) for s in soft_list))
        buf = np.zeros((self.n, cap), dtype=np.int16)
        counts = np.zeros(self.n, dtype=np.int32)
        for c, s in enumerate(soft_list):
            buf[c, :len(s)] = s; counts[c] = len(s)
        _check(lib().jaero_pchannel_process_softbits(self.h, _p(buf), cap, _p(counts)))

    def tick(self, batch=None):
        _check(lib().jaero_pchannel_tick(self.h, batch.h if batch is not None else None))

    def lost_signal(self, batch=None, channel=-1):
        """AeroL::SignalStatusSlot(false) -> LostSignal()"""
        _check(lib().jaero_pchannel_lost_signal(self.h, batch.h if batch is not None else None, channel))

    def write_batch(self, batch, pcm):
        """writeData with this AeroL attached as the reference wires them (cut at every estimator trigger)"""
        pcm = np.ascontiguousarray(pcm)
        assert pcm.dtype == np.int16 and pcm.ndim == 2 and pcm.shape[0] == self.n
        _check(lib().jaero_pchannel_write_batch(self.h, batch.h, _p(pcm), pcm.shape[1], pcm.strides[0] // 2 if pcm.shape[0] > 1 else pcm.shape[1]))

    def read_sus(self):
        """-> per channel: (bytes[n,12], crc_ok[n], index_in_frame[n], frame[n])"""
        out = np.zeros((self.n, self.su_cap, 16), dtype=np.uint8)
        counts = np.zeros(self.n, dtype=np.int32)
        _check(lib().jaero_pchannel_read_sus(self.h, _p(out), self.su_cap, _p(counts)))
        res = []
        for c in range(self.n):
            r = out[c, :counts[c]]
            res.append((r[:, :12].copy(), r[:, 12].astype(np.int32), r[:, 13].astype(np.int32),
                        r[:, 14].astype(np.int32) | (r[:, 15].astype(np.int32) << 8)))
        return res

    def read_sus_raw(self, out=None, counts=None):
        """The C-ABI call without per-channel Python objects: (records[n_channels, su_cap, 16] uint8, counts[n_channels]);
        record = 12 SU bytes, crc_ok, index in frame, frame number (lo, hi)."""
        if out is None:
            out = np.empty((self.n, self.su_cap, 16), dtype=np.uint8)
        if counts is None:
            counts = np.zeros(self.n, dtype=np.int32)
        _check(lib().jaero_pchannel_read_sus(self.h, _p(out), self.su_cap, _p(counts)))
        return out, counts

    def discard_sus(self):
        _check(lib().jaero_pchannel_discard_sus(self.h))

    def stats(self):
        dcd = np.zeros(self.n, dtype=np.int32); tot = np.zeros(self.n, dtype=np.int64); ok = np.zeros(self.n, dtype=np.int64)
        _check(lib().jaero_pchannel_get_stats(self.h, _p(dcd), _p(tot), _p(ok)))
        return dcd, tot, ok

    @property
    def launches(self):
        return lib().jaero_pchannel_launch_count(self.h)

    def close(self):
        if self.h:
            lib().jaero_pchannel_destroy(self.h); self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class BurstStatus(ctypes.Structure):
    _fields_ = [(n, ctypes.c_double) for n in
                ("mixer2_freq", "mixer2_wtptr", "center_freq", "st_freq", "st_wtptr", "agc", "mse", "ebno", "vol_gain",
                 "rotator_freq", "n_sig_true", "n_sig_false", "cntr", "startstop", "last_burst_ebno", "n_ebno_emits")]


class BurstMskBatch:
    """n_channels independent burst MSK demodulators (BurstMskDemodulator, 600 / 1200 bps R/T channels)."""

    def __init__(self, n_channels, fb=1200.0, Fs=48000.0, freq_center=1000.0, lockingbw=1800.0, signalthreshold=0.6, device=0):
        if n_channels <= 0:
            raise JaeroError("n_channels must be positive")
        s = Settings(KIND_MSK, 13, freq_center, lockingbw, fb, Fs, signalthreshold, 1, 0, 0, 1)
        self.h = ctypes.c_void_p()
        self.n = n_channels
        self.soft_cap = max(4096, int(2 * fb) + 64)
        _check(lib().jaero_burst_msk_create(ctypes.byref(s), n_channels, device, ctypes.byref(self.h)))

    def write(self, pcm):
        pcm = np.asarray(pcm)
        assert pcm.dtype == np.int16 and pcm.ndim == 2 and pcm.shape[0] == self.n
        if not pcm.flags.c_contiguous:
            pcm = np.ascontiguousarray(pcm)
        _check(lib().jaero_burst_write(self.h, _p(pcm), pcm.shape[1], pcm.strides[0] // 2 if pcm.shape[0] > 1 else pcm.shape[1]))

    def write_device(self, dev_ptr, n_samples, stride):
        """writeData from a DEVICE buffer [n_channels][stride] int16"""
        _check(lib().jaero_burst_write_device(self.h, ctypes.c_void_p(dev_ptr), n_samples, stride))

    def read_softbits(self):
        out = np.zeros((self.n, self.soft_cap), dtype=np.int16)
        counts = np.zeros(self.n, dtype=np.int32)
        _check(lib().jaero_burst_read_softbits(self.h, _p(out), self.soft_cap, _p(counts)))
        return [out[c, :counts[c]].copy() for c in range(self.n)]

    def set_dcd(self, dcd, channel=-1):
        _check(lib().jaero_burst_set_dcd(self.h, channel, int(dcd)))

    def status(self):
        arr = (BurstStatus * self.n)()
        _check(lib().jaero_burst_get_status_all(self.h, ctypes.cast(arr, ctypes.c_void_p)))
        return [{f[0]: getattr(arr[c], f[0]) for f in BurstStatus._fields_} for c in range(self.n)]

    def sync(self):
        _check(lib().jaero_burst_sync(self.h))

    @property
    def launches(self):
        return lib().jaero_burst_launch_count(self.h)

    def close(self):
        if self.h:
            lib().jaero_burst_destroy(self.h); self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class BurstOqpskBatch(BurstMskBatch):
    """n_channels independent burst OQPSK demodulators (BurstOqpskDemodulator, 10500 bps bursts)."""

    def __init__(self, n_channels, fb=10500.0, Fs=48000.0, freq_center=8000.0, lockingbw=10500.0, signalthreshold=0.6, sql=False, device=0):
        if n_channels <= 0:
            raise JaeroError("n_channels must be positive")
        s = Settings(KIND_OQPSK, 13, freq_center, lockingbw, fb, Fs, signalthreshold, 1, int(bool(sql)), 0, 1)
        self.h = ctypes.c_void_p()
        self.n = n_channels
        self.soft_cap = max(4096, int(2 * fb) + 64)
        _check(lib().jaero_burst_oqpsk_create(ctypes.byref(s), n_channels, device, ctypes.byref(self.h)))


class RTChannelBatch:
    """R/T burst channel layer for n_channels streams: soft bits (with -1 start-of-burst markers) -> R / T packets."""
    RECORD = 400

    def __init__(self, n_channels, fb, device=0):
        if n_channels <= 0:
            raise JaeroError("n_channels must be positive")
        self.h = ctypes.c_void_p()
        self.n = n_channels
        _check(lib().jaero_rt_create(float(fb), n_channels, device, ctypes.byref(self.h)))

    def process(self, soft_list):
        """soft_list: one int16 array per channel."""
        cap = max(1, max(len(s) for s in soft_list))
        buf = np.zeros((self.n, cap), dtype=np.int16)
        counts = np.zeros(self.n, dtype=np.int32)
        for c, s in enumerate(soft_list):
            buf[c, :len(s)] = s; counts[c] = len(s)
        _check(lib().jaero_rt_process_softbits(self.h, _p(buf), cap, _p(counts)))

    def process_burst(self, burst_batch):
        _check(lib().jaero_rt_process_burst(self.h, burst_batch.h))

    def tick(self):
        _check(lib().jaero_rt_tick(self.h))

    def set_vector_mode(self, on=True):
        """AeroL::Decode's mid-vector return on burst time-out (aerol.cpp:2018-2027)"""
        _check(lib().jaero_rt_set_vector_mode(self.h, int(bool(on))))

    def read_packets(self, cap=8):
        out = np.zeros((self.n, cap, self.RECORD), dtype=np.uint8)
        counts = np.zeros(self.n, dtype=np.int32)
        _check(lib().jaero_rt_read_packets(self.h, _p(out), cap, _p(counts)))
        res = []
        for c in range(self.n):
            pk = []
            for k in range(counts[c]):
                hdr = out[c, k, :16].view(np.int32)
                pk.append(dict(type=int(hdr[0]), nsus=int(hdr[1]), start_bit=int(hdr[3]), bytes=out[c, k, 16:16 + int(hdr[2])].copy()))
            res.append(pk)
        return res

    def stats(self):
        tr = np.zeros(self.n, dtype=np.int32); bad = np.zeros(self.n, dtype=np.int32); dcd = np.zeros(self.n, dtype=np.int32)
        _check(lib().jaero_rt_get_stats(self.h, _p(tr), _p(bad), _p(dcd)))
        return tr, bad, dcd

    @property
    def launches(self):
        return lib().jaero_rt_launch_count(self.h)

    def close(self):
        if self.h:
            lib().jaero_rt_destroy(self.h); self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class CChannelBatch:
    """C-channel (8400 bps) frame layer: soft bits -> per frame three sub-band signal units (+CRC) and 25 x 12 voice bytes."""
    RECORD = 352

    def __init__(self, n_channels, device=0):
        if n_channels <= 0:
            raise JaeroError("n_channels must be positive")
        self.h = ctypes.c_void_p()
        self.n = n_channels
        _check(lib().jaero_cchannel_create(n_channels, device, ctypes.byref(self.h)))

    def process(self, soft_list):
        cap = max(1, max(len(s) for s in soft_list))
        buf = np.zeros((self.n, cap), dtype=np.int16)
        counts = np.zeros(self.n, dtype=np.int32)
        for c, s in enumerate(soft_list):
            buf[c, :len(s)] = s; counts[c] = len(s)
        _check(lib().jaero_cchannel_process_softbits(self.h, _p(buf), cap, _p(counts)))

    def process_batch(self, batch):
        _check(lib().jaero_cchannel_process_batch(self.h, batch.h))

    def tick(self, batch=None):
        _check(lib().jaero_cchannel_tick(self.h, batch.h if batch is not None else None))

    def lost_signal(self, batch=None, channel=-1):
        _check(lib().jaero_cchannel_lost_signal(self.h, batch.h if batch is not None else None, channel))

    def write_batch(self, batch, pcm):
        pcm = np.ascontiguousarray(pcm)
        assert pcm.dtype == np.int16 and pcm.ndim == 2 and pcm.shape[0] == self.n
        _check(lib().jaero_cchannel_write_batch(self.h, batch.h, _p(pcm), pcm.shape[1], pcm.strides[0] // 2 if pcm.shape[0] > 1 else pcm.shape[1]))

    def read_frames(self, cap=8):
        """per channel: (su[n,3,12], crc_ok[n,3], voice[n,300], frame[n])"""
        out = np.zeros((self.n, cap, self.RECORD), dtype=np.uint8)
        counts = np.zeros(self.n, dtype=np.int32)
        _check(lib().jaero_cchannel_read_frames(self.h, _p(out), cap, _p(counts)))
        res = []
        for c in range(self.n):
            r = out[c, :counts[c]]
            su = r[:, :48].reshape(-1, 3, 16)
            res.append((su[:, :, :12].copy(), su[:, :, 12].astype(np.int32), r[:, 48:348].copy(), r[:, 348:352].copy().view(np.int32).reshape(-1)))
        return res

    def stats(self):
        dcd = np.zeros(self.n, dtype=np.int32); tot = np.zeros(self.n, dtype=np.int64); ok = np.zeros(self.n, dtype=np.int64)
        _check(lib().jaero_cchannel_get_stats(self.h, _p(dcd), _p(tot), _p(ok)))
        return dcd, tot, ok

    @property
    def launches(self):
        return lib().jaero_cchannel_launch_count(self.h)

    def close(self):
        if self.h:
            lib().jaero_cchannel_destroy(self.h); self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class IngestRouter:
    """ZMQ-style [topic][uint32 rate][int16 PCM] messages -> per-channel staging -> DemodBatch.write (host side, no libzmq)."""

    def __init__(self, topics, sample_rate=48000, capacity_samples=192000):
        self.n = len(topics)
        arr = (ctypes.c_char_p * self.n)(*[t.encode() if isinstance(t, str) else t for t in topics])
        self.h = ctypes.c_void_p()
        _check(lib().jaero_ingest_create(self.n, arr, int(sample_rate), int(capacity_samples), ctypes.byref(self.h)))

    def message(self, topic, rate_frame, pcm_frame):
        """three frames of one multipart message (bytes); returns the channel index"""
        topic = topic.encode() if isinstance(topic, str) else bytes(topic)
        pcm_frame = bytes(pcm_frame)
        buf = ctypes.create_string_buffer(pcm_frame, len(pcm_frame))
        rc = lib().jaero_ingest_message(self.h, topic, len(topic), bytes(rate_frame), len(rate_frame), ctypes.cast(buf, ctypes.c_void_p), len(pcm_frame))
        if rc < 0:
            raise JaeroError(lib().jaero_last_error().decode())
        return rc

    @property
    def available(self):
        return int(lib().jaero_ingest_available(self.h))

    def flush(self, batch, n=None):
        n = self.available if n is None else n
        _check(lib().jaero_ingest_flush(self.h, batch.h, n))
        return n

    def close(self):
        if self.h:
            lib().jaero_ingest_destroy(self.h); self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Reassembler:
    """Per-channel ISU/SSU reassembly + ACARS parsing + defragmentation (host side; mirrors the reference's ISUData,
    RISUData, ParserISU and ACARSDefragmenter, JAERO/aerol.cpp:4-487). Feed CRC-valid signal units only."""

    COMPLETE, MISSING, PARSED = 1, 2, 4

    def __init__(self):
        self.h = ctypes.c_void_p()
        _check(lib().jaero_reasm_create(ctypes.byref(self.h)))

    def reset(self):
        _check(lib().jaero_reasm_reset(self.h))

    def short_frame(self):
        _check(lib().jaero_reasm_short_frame(self.h))

    def push_su(self, su, downlink=False):
        su = bytes(bytearray(su))
        if len(su) < 10:
            raise ValueError("a signal unit has at least 10 bytes")
        return lib().jaero_reasm_push_su(self.h, su, int(downlink))

    def push_r(self, info, downlink=True):
        info = bytes(bytearray(info))
        if len(info) < 17:
            raise ValueError("an R-channel packet has at least 17 bytes")
        return lib().jaero_reasm_push_r(self.h, info, int(downlink))

    def push_t_packet(self, info, n_sus):
        info = bytes(bytearray(info))
        if len(info) < 6 + 12 * n_sus:
            raise ValueError("T packet shorter than its SU count")
        return lib().jaero_reasm_push_t_packet(self.h, info, int(n_sus))

    def pop_all(self):
        """list of dicts; text is bytes (message text, hex dump for non-ACARS user data, or the error string)"""
        out = []
        rec = AcarsRecord(); cap = 4096; buf = ctypes.create_string_buffer(cap)
        while True:
            n = lib().jaero_reasm_pop(self.h, ctypes.byref(rec), buf, cap)
            if n == -1:
                break
            if n == -2:
                cap = int(rec.text_len) + 1; buf = ctypes.create_string_buffer(cap)
                continue
            if n < 0:
                raise JaeroError("jaero_reasm_pop failed")
            f = rec.flags
            out.append(dict(kind=rec.kind, aesid=rec.aes_id, gesid=rec.ges_id, qno=rec.qno, refno=rec.refno, seqno=rec.seqno,
                            nooct=rec.last_octets, mode=rec.mode, tak=rec.tak, bi=rec.block_id,
                            nonacars=bool(f & 1), downlink=bool(f & 2), valid=bool(f & 4), hastext=bool(f & 8), moretocome=bool(f & 16),
                            label=bytes(rec.label[:rec.label_len]), reg=bytes(rec.reg[:rec.reg_len]), text=buf.raw[:n],
                            userdata_len=rec.userdata_len))
        return out

    def stats(self):
        v = (ctypes.c_uint64 * 4)()
        a = ctypes.addressof(v)
        _check(lib().jaero_reasm_get_stats(self.h, a, a + 8, a + 16, a + 24))
        return dict(isus=v[0], messages=v[1], errors=v[2], missing=v[3])

    def close(self):
        if self.h:
            lib().jaero_reasm_destroy(self.h); self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _chan_settings(input_rate, output_rate, audio_hz, passband_hz, iq_format, gain):
    if iq_format not in IQ_FORMATS:
        raise JaeroError("iq_format must be one of %s" % sorted(IQ_FORMATS))
    return ChanSettings(IQ_FORMATS[iq_format], 0, float(input_rate), float(output_rate), float(audio_hz), float(passband_hz), float(gain))


def channelizer_taps(input_rate, output_rate=48000.0, audio_hz=12000.0, passband_hz=12000.0, iq_format="cs16", gain=1.0):
    """The channelizer's low-pass prototype h[0..T-1] (float64, designed at L * input_rate, sum L: unity DC gain in each
    polyphase branch), designed on the host; no device needed."""
    s = _chan_settings(input_rate, output_rate, audio_hz, passband_hz, iq_format, gain)
    T = lib().jaero_chan_taps(ctypes.byref(s), None, 0)
    if T < 0:
        _check(T)
    h = np.zeros(T, dtype=np.float64)
    lib().jaero_chan_taps(ctypes.byref(s), _p(h), T)
    return h


def channelizer_ratio(input_rate, output_rate=48000.0, audio_hz=12000.0, passband_hz=12000.0, iq_format="cs16", gain=1.0):
    """(L, M) with output_rate / input_rate = L/M in lowest terms, as the channelizer accepts it (L <= 64, M >= 2L; L = 1 for
    an integer ratio); validates every setting as channelizer_taps does. No device needed."""
    s = _chan_settings(input_rate, output_rate, audio_hz, passband_hz, iq_format, gain)
    Lr, Mr = ctypes.c_int(), ctypes.c_int()
    _check(lib().jaero_chan_ratio(ctypes.byref(s), ctypes.byref(Lr), ctypes.byref(Mr)))
    return Lr.value, Mr.value


class Channelizer:
    """One wideband complex IQ stream -> one real int16 audio row per channel (channel c's carrier moved to audio_hz at
    output_rate), on the device. The rows feed DemodBatch.write_device(ptr, n, stride) as they are (see output_device).
    ratio is (L, M), output_rate / input_rate = L/M; D is the integer ratio M when L = 1, else None."""

    def __init__(self, offsets_hz, input_rate, output_rate=48000.0, audio_hz=12000.0, passband_hz=12000.0, iq_format="cs16",
                 gain=1.0, device=0):
        s = _chan_settings(input_rate, output_rate, audio_hz, passband_hz, iq_format, gain)
        off = np.ascontiguousarray(np.atleast_1d(np.asarray(offsets_hz, dtype=np.float64)))
        self.h = ctypes.c_void_p()
        self.n = len(off)
        self.iq_format = iq_format
        _check(lib().jaero_chan_create(ctypes.byref(s), self.n, _p(off), device, ctypes.byref(self.h)))
        self.ratio = channelizer_ratio(input_rate, output_rate, audio_hz, passband_hz, iq_format, gain)
        self.D = self.ratio[1] if self.ratio[0] == 1 else None

    def write(self, iq):
        """iq: host array [n, 2] of int16 (cs16) or uint8 (cu8) I, Q pairs."""
        iq = np.ascontiguousarray(iq)
        want = np.int16 if self.iq_format == "cs16" else np.uint8
        if iq.dtype != want or iq.ndim != 2 or iq.shape[1] != 2:
            raise JaeroError("write expects a [n, 2] %s array" % np.dtype(want).name)
        _check(lib().jaero_chan_write(self.h, _p(iq), iq.shape[0]))

    def write_device(self, dev_ptr, n_iq):
        """n_iq complex samples already in this GPU's memory (interleaved I, Q in the handle's format)."""
        _check(lib().jaero_chan_write_device(self.h, ctypes.c_void_p(dev_ptr), int(n_iq)))

    def output_device(self):
        """(device pointer, samples per channel, channel stride) of the rows the last write produced; valid until the next write."""
        a, n, st = ctypes.c_void_p(), ctypes.c_size_t(), ctypes.c_size_t()
        _check(lib().jaero_chan_output_device(self.h, ctypes.byref(a), ctypes.byref(n), ctypes.byref(st)))
        return a.value, n.value, st.value

    def read(self):
        """int16 [n_channels, n] copy of the rows the last write produced (synchronises)."""
        _, n, _ = self.output_device()
        out = np.zeros((self.n, max(n, 1)), dtype=np.int16)
        got = ctypes.c_size_t()
        _check(lib().jaero_chan_read(self.h, _p(out), out.shape[1], ctypes.byref(got)))
        return out[:, :got.value]

    def set_stream(self, cuda_stream):
        _check(lib().jaero_chan_set_stream(self.h, ctypes.c_void_p(cuda_stream)))

    def sync(self):
        _check(lib().jaero_chan_sync(self.h))

    @property
    def launches(self):
        return lib().jaero_chan_launch_count(self.h)

    def close(self):
        if self.h:
            lib().jaero_chan_destroy(self.h); self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
