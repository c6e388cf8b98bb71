#!/usr/bin/env python
"""bench.py — benchmarks of the jaero_b200 hot path.

Default workload `oqpsk10500` (BASELINE.json configs[2], the one the metric is quoted on): 4096 concurrent continuous
10.5 kbps OQPSK P-channels per GPU, synthetic real-passband int16 @48 kHz (Eb/N0 = 10 dB), each step = 1 s of signal per
channel through  demodulator (K1a) + coarse frequency estimator (K2) + P-channel framing + fused de-interleave/Viterbi
(K5) + descramble + CRC  with DCD fed back. Metric: Msamples/s (one sample = one int16 input sample of one channel);
channels@RT = samples/s / 48000.

  python bench.py --gpus N --steps K --warmup W            our CUDA path (one process per GPU under torchrun)
  python bench.py --impl reference ...                      the reference's own CPU path on this box's host cores
  python bench.py --workload msk1200                        BASELINE configs[1]: 1024-channel continuous 1200 bps MSK, Eb/N0 8 dB
  python bench.py --workload burst1200x2048                 BASELINE configs[3]: the burst recording x2048, random frequency offsets
  python bench.py --workload mix16384 [--scaling strong]    BASELINE configs[4]: 10.5k OQPSK + 8400 bps C-channel mix, sharded
  python bench.py ... --dump-outputs DIR                    also write what the last timed step decoded as DIR/<name>.npy

Prints ONE JSON line (rank 0). `value` = device-timed, input resident in HBM; `e2e` = through the C ABI with HOST
buffers (H2D of the PCM and D2H of the decoded signal units inside the timed region).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FS = 48000
STEP_SAMPLES = 48000                  # 1 s of signal per channel per step
# Algorithmic bytes per input sample and channel (SURVEY.md section 8(d), DESIGN.md section 4): what one pass must move at least
ALG_K1A = 66.2                        # 2 PCM + 16 AGC ring + 32 EbNo rings + 16 estimator-ring write + 0.22 soft bits
ALG_K2 = 128.0                        # estimator frame traffic: 32*nfft bytes per nfft/4 samples
ALG_STEP = 194.2                      # the whole step (K1a + K2)
ALG_MSK = 2 + 16 + 32 + 16 + 128 + 0.05   # same accounting for the MSK path (nfft 8192 per 2048 samples -> 128 B/sample)

MODES = {
    "oqpsk10500": dict(kind="oqpsk", fb=10500, fc0=8000, fc_span=500, lockingbw=10500, ebn0=10.0, channels=4096, frames=2,
                       metric="IQ Msamples/s (10.5k OQPSK demod + Viterbi)", alg=ALG_K1A, kernel="oqpsk_pipe_kernel",
                       label="4096-channel 10.5 kbps continuous OQPSK + Viterbi, synthetic real-passband int16 @48 kHz (BASELINE configs[2])"),
    "msk1200": dict(kind="msk", fb=1200, fc0=2000, fc_span=200, lockingbw=1800, ebn0=8.0, channels=1024, frames=1,
                    metric="IQ Msamples/s (1200 bps MSK demod + Viterbi)", alg=ALG_MSK - 128.0, kernel="msk_pipe_kernel",
                    label="1024-channel 1200 bps continuous MSK + Viterbi, synthetic real-passband int16 @48 kHz, Eb/N0 8 dB (BASELINE configs[1])"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="oqpsk10500", choices=["oqpsk10500", "msk1200", "burst1200x2048", "mix16384"])
    ap.add_argument("--channels", type=int, default=0, help="channels per GPU (0 = the workload's own count)")
    ap.add_argument("--ebn0", type=float, default=None)
    ap.add_argument("--cpu-seconds", type=float, default=40.0, help="seconds of signal per channel for the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-saturation", action="store_true", help="skip the 8192/16384/32768-channel saturation block (N=1, default workload)")
    ap.add_argument("--streams", type=int, default=1, help="continuous workloads: split a GPU's channels into this many batches, each on its own CUDA stream "
                    "(the demodulator epoch of one batch then overlaps the estimator epoch of another)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"], help="mix16384: weak = 2048 channels per GPU, strong = 16384 in total")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="continuous workloads: write what the last timed step decoded (signal units, CRC flags, DCD, loop state) "
                    "as DIR/<name>.npy, so that two builds can be compared output for output")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "ours" or a.workload not in MODES):
        ap.error("--dump-outputs applies to --impl ours with a continuous workload (%s)" % ", ".join(MODES))
    return a


# ----------------------------------------------------------------------------- synthetic input
def base_envelopes(mode, n_base, seed):
    """n_base distinct, seamlessly loopable 1 s complex envelopes (numpy, rank 0)."""
    from jaero_b200 import synth
    m = MODES[mode]
    envs = []
    for k in range(n_base):
        if m["kind"] == "oqpsk":
            bits = synth.pchannel_bits(m["fb"], m["frames"], seed=seed + k)
            envs.append(synth.oqpsk_envelope(bits, m["fb"], FS))
        else:
            bits = synth.pchannel_bits(m["fb"], m["frames"], seed=seed + k, loop=True, even_parity=True)
            envs.append(synth.msk_envelope(bits, m["fb"], FS))
    return np.stack(envs).astype(np.complex64)


def make_pcm_gpu(mode, envs_t, ch0, n_ch, ebn0_db, device):
    """Per-channel real passband int16 on the GPU: base envelope (c % B) with a circular delay, integer-Hz carrier
    fc0 + U(-span, span), random phase, AWGN at Eb/N0, RMS 0.2 FS. Seeds depend on the GLOBAL channel index."""
    import torch
    m = MODES[mode]
    B, L = envs_t.shape
    out = torch.empty((n_ch, L), dtype=torch.int16, device=device)
    n = torch.arange(L, device=device, dtype=torch.float64)
    fcs = np.zeros(n_ch)
    for a in range(0, n_ch, 256):
        mm = min(256, n_ch - a)
        g = torch.Generator(device="cpu"); g.manual_seed(0x4A4145524F + ch0 + a)
        delay = torch.randint(0, L, (mm,), generator=g)
        fc = m["fc0"] + torch.randint(-m["fc_span"], m["fc_span"] + 1, (mm,), generator=g).to(torch.float64)
        ph = torch.rand((mm,), generator=g, dtype=torch.float64) * 2 * np.pi
        fcs[a:a + mm] = fc.numpy()
        idx = (torch.arange(L).unsqueeze(0) - delay.unsqueeze(1)) % L
        k = (torch.arange(ch0 + a, ch0 + a + mm) % B)
        env = envs_t[k.to(device).unsqueeze(1), idx.to(device)]
        arg = (2 * np.pi * fc.to(device).unsqueeze(1) * n.unsqueeze(0) / FS + ph.to(device).unsqueeze(1))
        x = (env.real.to(torch.float64) * torch.cos(arg) - env.imag.to(torch.float64) * torch.sin(arg)).to(torch.float32)
        ps = (x * x).mean(dim=1, keepdim=True)
        if ebn0_db is not None:
            n0 = ps * (FS / m["fb"]) / (10 ** (ebn0_db / 10.0))
            gg = torch.Generator(device=device); gg.manual_seed(12345 + ch0 + a)
            x = x + torch.randn(x.shape, generator=gg, device=device) * torch.sqrt(n0 / 2.0)
        x = x * (0.2 / torch.sqrt((x * x).mean(dim=1, keepdim=True)))
        out[a:a + mm] = torch.clamp(torch.round(x * 32767.0), -32768, 32767).to(torch.int16)
    return out, fcs


def offset_replicas_gpu(base_i16, offsets_hz, device):
    """Re{hilbert(x) e^(j 2 pi df n / Fs)} -> int16, one row per offset (SURVEY.md section 8(d) cfg 4); torch twin of
    jaero_b200.synth.offset_replicas."""
    import torch
    x = base_i16.to(device=device, dtype=torch.float64)
    n = x.numel()
    X = torch.fft.fft(x)
    h = torch.zeros(n, dtype=torch.float64, device=device)
    h[0] = 1.0
    if n % 2 == 0:
        h[n // 2] = 1.0; h[1:n // 2] = 2.0
    else:
        h[1:(n + 1) // 2] = 2.0
    an = torch.fft.ifft(X * h)
    t = torch.arange(n, device=device, dtype=torch.float64) / FS
    out = torch.empty((len(offsets_hz), n), dtype=torch.int16, device=device)
    for r0 in range(0, len(offsets_hz), 64):
        df = torch.as_tensor(np.asarray(offsets_hz[r0:r0 + 64]), dtype=torch.float64, device=device).unsqueeze(1)
        ph = 2 * np.pi * df * t.unsqueeze(0)
        y = an.real.unsqueeze(0) * torch.cos(ph) - an.imag.unsqueeze(0) * torch.sin(ph)
        out[r0:r0 + y.shape[0]] = torch.clamp(torch.round(y), -32768, 32767).to(torch.int16)
    return out


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi polled every 100 ms from BEFORE the warm-up (its start-up takes longer than a short timed region);
    only the rows received between mark_begin() and stop() - i.e. during the timed region - are reported."""

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index
        self.t_begin = None

    def mark_begin(self):
        self.t_begin = time.perf_counter()

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        t_end = time.perf_counter()
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        t0 = self.t_begin if self.t_begin is not None else 0.0
        for t, r in self.rows:
            if t < t0 or t > t_end + 0.05:
                continue
            f = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------- CPU reference arm
def usable_cores():
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:                                                     # cgroup v2 / v1 CPU quota
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(float(q) / float(per))))
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()); per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, q // per))
        except Exception:
            pass
    return n


def _cpu_worker(args):
    """One host core: the reference's demodulator (oracle/_ref, verbatim build) or the restated port, followed by the restated
    AeroL frame layer (frame sync, de-interleave, Viterbi, CRC) with DCD fed back — the same work per sample as the GPU
    pipeline. `pcm` is one period of a seamlessly looping signal, repeated n_loops times (or a recording played once).
    Returns (samples, seconds, su_total, su_ok)."""
    impl, kind, fb, lockingbw, pcm, n_loops, fc = args
    from oracle import ref, restated
    if kind in ("burst_msk",):
        kw = dict(fb=float(fb), freq_center=float(fc), lockingbw=float(lockingbw), signalthreshold=0.6)
    else:
        kw = dict(fb=fb, freq_center=fc, lockingbw=lockingbw, fft_power=14 if kind == "oqpsk" else 13,
                  signalthreshold=0.65 if kind == "oqpsk" else 0.5, afc=(fb == 8400))
    d = ref.RefDemod(kind, **kw) if impl == "reference" else restated.OracleDemod(kind, **kw)
    if kind == "burst_msk":
        layer = restated.OracleRTChannel(fb)
    elif fb == 8400:
        layer = restated.OracleCChannel()
    else:
        layer = restated.OraclePChannel(fb)
    t0 = time.perf_counter()
    tot = ok = 0
    for s in range(n_loops):
        for a in range(0, len(pcm), 4800):                   # 100 ms writeData calls (BASELINE.md section 4)
            d.write(pcm[a:a + 4800])
            layer.process(d.take_soft())
            if kind != "burst_msk":
                d.set_dcd(int(layer.dcd))
        layer.update_dcd()
        if kind == "burst_msk":
            pk = layer.packets(); tot += len(pk); ok += len(pk)
        elif fb == 8400:
            _, o, _ = layer.take_frames(); tot += o.size; ok += int(o.sum())
        else:
            _, o, _ = layer.take_sus(); tot += len(o); ok += int(o.sum())
    return len(pcm) * n_loops, time.perf_counter() - t0, tot, ok


def cpu_reference_run(jobs, cores):
    """jobs: (kind, fb, lockingbw, pcm_row, n_loops, fc). One fresh process per job (the reference keeps function-local statics)."""
    import multiprocessing as mp
    from oracle import ref, restated
    impl = "reference" if ref.available() else "port"
    if impl == "port" and not restated.available():
        raise RuntimeError("neither oracle/_ref nor oracle/_build is built")
    t0 = time.perf_counter()
    with mp.get_context("spawn").Pool(cores) as pool:
        res = pool.map(_cpu_worker, [(impl,) + tuple(j) for j in jobs], chunksize=1)
    wall = time.perf_counter() - t0
    samples = sum(r[0] for r in res)
    # throughput of the box = samples / the time the busiest core needed; jobs are dealt one per core in rounds
    rounds = (len(jobs) + cores - 1) // cores
    busy = max(r[1] for r in res) * rounds if rounds > 1 else max(r[1] for r in res)
    return impl, samples, busy, wall, sum(r[2] for r in res), sum(r[3] for r in res)


def cpu_baseline_block(jobs, cores, what):
    """The bounded CPU sample printed next to the GPU numbers: one core alone first (warms caches, gives the per-core figure)."""
    _, s1, b1, _, _, _ = cpu_reference_run(jobs[:1], 1)
    impl, samples, busy, wall, tot, ok = cpu_reference_run(jobs, cores)
    return {"value": samples / busy / 1e6, "unit": "Msamples/s", "cores": cores, "kind": impl, "single_core_value": s1 / b1 / 1e6,
            "sample": what, "cpu_seconds_busy": busy, "su_total": tot, "su_crc_ok": ok}


# ----------------------------------------------------------------------------- helpers
def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def ncu_traffic_bytes(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of `kernel`, from this round's committed `ncu --set full`
    capture profiles/r02_<kernel>_full_raw.csv (None if that capture is absent: never a stale round's number)."""
    import csv
    path = os.path.join(ROOT, "profiles", "r02_%s_full_raw.csv" % kernel)
    try:
        rows = list(csv.reader(open(path)))
        hdr, units, row = rows[0], rows[1], rows[2]
        tot = 0.0
        for k in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            i = hdr.index(k)
            tot += float(row[i].replace(",", "")) * {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}[units[i]]
        return tot, os.path.relpath(path, ROOT)
    except Exception:
        return None, None


class Pipeline:
    """One continuous-mode batch + its frame layer on one GPU, with the PCM of one step resident in HBM."""

    def __init__(self, mode, C, ch0, ebn0, envs_t, dev, local, stream=None):
        import jaero_b200
        m = MODES[mode]
        self.m, self.C = m, C
        self.pcm, self.fcs = make_pcm_gpu(mode, envs_t, ch0, C, ebn0, dev)
        self.batch = jaero_b200.DemodBatch(m["kind"], C, fb=m["fb"], freq_center=self.fcs, lockingbw=m["lockingbw"], afc=False, report_ebno=True, device=local)
        self.layer = jaero_b200.PChannelBatch(C, m["fb"], device=local)
        if stream is not None:
            self.batch.set_stream(stream.cuda_stream)      # demod segments, estimator, frame layer, Viterbi all launch here
        self.stream = stream
        self.stride = self.pcm.stride(0)

    def step_device(self, keep_sus=False):
        self.batch.write_device(self.pcm.data_ptr(), STEP_SAMPLES, self.stride)
        self.layer.process_batch(self.batch)
        self.layer.tick(self.batch)
        if not keep_sus:
            self.layer.discard_sus()      # results stay on the device for the HBM-resident measurement

    @property
    def launches(self):
        return self.batch.launches + self.layer.launches

    def close(self):
        self.batch.close(); self.layer.close()


def timed_steps(pipes, stream, steps, warmup, rank, local, dev, keep_last=False):
    """W warm-up steps, then exactly K steps between CUDA events on the launching stream; max over ranks.
    keep_last: the signal units of the last timed step stay queued for read_sus instead of being discarded."""
    import torch
    from jaero_b200 import shard
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    for _ in range(max(3, warmup)):
        for p in pipes:
            p.step_device()
    torch.cuda.synchronize(); shard.barrier()
    l0 = sum(p.launches for p in pipes)
    for p in pipes:
        p.batch.set_profiling(True); p.batch.get_profile()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    others = [p.stream for p in pipes if getattr(p, "stream", None) is not None and p.stream is not stream]
    torch.cuda.synchronize(); shard.barrier()
    clocks.mark_begin()
    e0.record(stream)
    for so in others:
        so.wait_event(e0)                 # no batch starts before e0 ...
    for k in range(steps):
        for p in pipes:
            p.step_device(keep_sus=keep_last and k == steps - 1)
    for so in others:
        ej = torch.cuda.Event(); ej.record(so); stream.wait_event(ej)   # ... and e1 fires when every batch is done
    e1.record(stream)
    torch.cuda.synchronize(); shard.barrier()
    ms_local = e0.elapsed_time(e1)
    ms = shard.reduce_max(ms_local, device=dev)
    launches = sum(p.launches for p in pipes) - l0
    profs = []
    for p in pipes:
        profs.append(p.batch.get_profile()); p.batch.set_profiling(False)
    clk = clocks.stop() if rank == 0 else None
    return ms, ms_local, launches, profs, clk


def roofline_block(mode, prof, C, ms_local, peaks):
    m = MODES[mode]
    peak = float(peaks.get("hbm_gbs", 6650.0))
    seg_s, cfe_s = prof["segment_ms"] * 1e-3, prof["cfe_ms"] * 1e-3
    units = prof["samples"] * C                                   # channel-samples the timed launches processed
    ach = (m["alg"] * units) / seg_s / 1e9 if seg_s > 0 else 0.0
    ach2 = (ALG_K2 * units) / cfe_s / 1e9 if cfe_s > 0 else 0.0
    step_ach = ((m["alg"] + ALG_K2) * units) / (ms_local * 1e-3) / 1e9
    traffic, src = ncu_traffic_bytes(m["kernel"])
    return {"bound": "hbm", "kernel": m["kernel"], "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
            "traffic": traffic, "traffic_source": src,
            "peak_source": "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)",
            "alg_bytes_per_sample": m["alg"], "avg_launch_ms": prof["segment_ms"] / max(1, prof["segment_launches"]),
            "launches": prof["segment_launches"], "share_of_step": prof["segment_ms"] / ms_local,
            "kernels": [
                {"kernel": "cfe_cluster_kernel+cfe_search_kernel" if mode == "oqpsk10500" else "cfe_col/row kernels", "alg_bytes_per_sample": ALG_K2,
                 "achieved": ach2, "frac": ach2 / peak, "avg_epoch_ms": prof["cfe_ms"] / max(1, prof["cfe_runs"]), "share_of_step": prof["cfe_ms"] / ms_local},
                {"kernel": "whole step (all kernels)", "alg_bytes_per_sample": m["alg"] + ALG_K2, "achieved": step_ach, "frac": step_ach / peak}],
            "note": "per-channel fp64 feedback loop: bound by dependent-issue latency, not HBM (DESIGN.md section 5); K1a's own algorithmic bytes exclude the estimator's frame traffic, which is K2's"}


DUMP_LIMIT = 64 << 20                 # bytes --dump-outputs may write


def dump_outputs(out_dir, pipes):
    """What the last timed step handed a caller of the P-channel path, one .npy per array (float32 / float64): the decoded
    signal units of every channel concatenated in channel order (su_*, channel index in su_channel, per-channel count in
    su_count), the DCD flag and cumulative SU counters per channel, and the demodulator's loop state per channel (state_*).
    If the signal units would exceed DUMP_LIMIT, a fixed seeded sample of channels is kept (listed in su_channels_kept)."""
    recs, counts = [], []
    for p in pipes:
        r, c = p.layer.read_sus_raw()
        recs.append(r); counts.append(c)
    rec = np.concatenate(recs); cnt = np.concatenate(counts).astype(np.int64)
    n_ch = len(cnt)
    keep = np.arange(n_ch)
    per_su = 4 * (12 + 4)                                         # float32 bytes + crc_ok, index, frame, channel
    if int(cnt.sum()) * per_su > DUMP_LIMIT // 2:
        n_keep = max(1, int(n_ch * (DUMP_LIMIT // 2) // (int(cnt.sum()) * per_su)))
        keep = np.sort(np.random.default_rng(0x4A4145).choice(n_ch, size=n_keep, replace=False))
    sel = np.concatenate([np.stack([np.full(cnt[c], c), np.arange(cnt[c])], 1) for c in keep]).astype(np.int64).reshape(-1, 2)
    r = rec[sel[:, 0], sel[:, 1]]
    st = [s for p in pipes for s in p.batch.status()]
    dcd, tot, ok = (np.concatenate([p.layer.stats()[i] for p in pipes]) for i in range(3))
    arrays = {"su_bytes": r[:, :12].astype(np.float32), "su_crc_ok": r[:, 12].astype(np.float32),
              "su_index_in_frame": r[:, 13].astype(np.float32),
              "su_frame": (r[:, 14].astype(np.int32) | (r[:, 15].astype(np.int32) << 8)).astype(np.float32),
              "su_channel": sel[:, 0].astype(np.float32), "su_count": cnt.astype(np.float32), "su_channels_kept": keep.astype(np.float32),
              "dcd": dcd.astype(np.float32), "su_total": tot.astype(np.float64), "su_crc_ok_total": ok.astype(np.float64)}
    for k in st[0]:
        if k != "reserved":
            arrays["state_" + k] = np.array([s[k] for s in st], dtype=np.float64)
    assert sum(v.nbytes for v in arrays.values()) <= DUMP_LIMIT
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


# ----------------------------------------------------------------------------- workloads
def run_continuous(a, mode):
    import torch
    from jaero_b200 import shard
    m = MODES[mode]
    cores = usable_cores()
    ebn0 = a.ebn0 if a.ebn0 is not None else m["ebn0"]
    if a.impl == "reference":
        rank = int(os.environ.get("RANK", "0"))
        n_gpus = max(a.gpus, int(os.environ.get("WORLD_SIZE", "1")))
        if rank != 0:
            return 0
        envs_t = torch.from_numpy(base_envelopes(mode, 16, 7))
        pcm, fcs = make_pcm_gpu(mode, envs_t, 0, cores, ebn0, "cpu")
        rows = [pcm[i].numpy().copy() for i in range(cores)]
        mk = lambda i, loops: (m["kind"], m["fb"], m["lockingbw"], rows[i], loops, float(fcs[i]))
        cpu_reference_run([mk(i, 1) for i in range(min(2, cores))], min(2, cores))            # warm the page cache / libm
        loops = max(1, a.steps) * 4
        impl, samples, busy, wall, tot, ok = cpu_reference_run([mk(i, loops) for i in range(cores)], cores)
        val = samples / busy / 1e6
        line = {"impl": "reference", "metric": m["metric"], "value": val, "unit": "Msamples/s",
                "n_gpus": n_gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": busy * 1e3 / max(1, a.steps),
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "channels_rt": val * 1e6 / FS,
                "config": {"workload": m["label"] + "; reference arm = bounded sample", "channels": cores, "seconds_per_step": 4.0, "ebn0_db": ebn0},
                "cpu_baseline": {"value": val, "unit": "Msamples/s", "cores": cores, "kind": impl,
                                 "sample": "%d channels x %d s, one process per core, 100 ms writeData calls, demod + P-channel decode" % (cores, loops)},
                "e2e": {"value": val, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "decode": {"su_total": tot, "su_crc_ok": ok}, "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    rank, local, world = shard.init_from_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    C = a.channels or m["channels"]
    ch0 = rank * C
    # shared source: base envelopes built on rank 0 and broadcast over NCCL/NVLink (the only collective besides reporting)
    envs_t = torch.zeros((16, STEP_SAMPLES), dtype=torch.complex64, device=dev)
    if rank == 0:
        envs_t.copy_(torch.from_numpy(base_envelopes(mode, 16, 7)))
    shard.broadcast_(torch.view_as_real(envs_t), 0)
    stream = torch.cuda.Stream(device=dev)          # a real (non-default) stream: handle 0 would mean "library's own stream"
    assert stream.cuda_stream != 0
    G = max(1, a.streams)
    if C % (32 * G):
        raise SystemExit("bench.py: --streams must divide the channel count into multiples of 32")
    Cg = C // G
    streams = [stream] + [torch.cuda.Stream(device=dev) for _ in range(G - 1)]
    pipes = [Pipeline(mode, Cg, ch0 + g * Cg, ebn0, envs_t, dev, local, streams[g]) for g in range(G)]
    pipe = pipes[0]
    torch.cuda.synchronize()
    ms, ms_local, launches, profs, clk = timed_steps(pipes, stream, a.steps, a.warmup, rank, local, dev, keep_last=bool(a.dump_outputs))
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, pipes)
    st = [p.layer.stats() for p in pipes]
    dcd, su_tot, su_ok = (np.concatenate([x[i] for x in st]) for i in range(3))
    total_samples = float(C) * STEP_SAMPLES * a.steps * world
    value = total_samples / (ms * 1e-3) / 1e6

    # ---- end-to-end through the C ABI with HOST buffers
    e2e = None
    if not a.no_e2e:
        hosts, bufs = [], []
        for p in pipes:
            host = torch.empty((Cg, STEP_SAMPLES), dtype=torch.int16).pin_memory()
            host.copy_(p.pcm.cpu())
            hosts.append(host.numpy())
            bufs.append((np.empty((Cg, p.layer.su_cap, 16), dtype=np.uint8), np.zeros(Cg, dtype=np.int32)))
        pch = pipe.layer

        def step_e2e():
            for p, h in zip(pipes, hosts):
                p.batch.write(h)                   # H2D of the step's PCM (pinned) inside the call
                p.layer.process_batch(p.batch)
                p.layer.tick(p.batch)
            for p, (su_buf, su_cnt) in zip(pipes, bufs):
                p.layer.read_sus_raw(su_buf, su_cnt)        # D2H of the decoded signal units + CRC flags (bulk records)
        step_e2e()
        torch.cuda.synchronize(); shard.barrier()
        t0 = time.perf_counter()
        for _ in range(a.steps):
            step_e2e()
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        ems = shard.reduce_max((t1 - t0) * 1e3, device=dev)
        e2e = {"value": total_samples / (ems * 1e-3) / 1e6, "unit": "Msamples/s", "h2d_bytes_per_step": int(C * STEP_SAMPLES * 2),
               "d2h_bytes_per_step": int(C * pch.su_cap * 16 + C * 120), "ms_per_step": ems / a.steps}

    tot = shard.reduce_sum([float(su_tot.sum()), float(su_ok.sum()), float(dcd.sum())], device=dev)
    peaks = load_peaks()
    prof = {k: sum(pr[k] for pr in profs) for k in profs[0]} if G > 1 else profs[0]
    if G > 1:
        prof["samples"] = profs[0]["samples"]; prof["batches"] = G
    roofline = roofline_block(mode, prof, C, ms_local, peaks)

    # ---- saturation: what the same pipeline reaches with more channels per GPU (the metric's 4096 leave most issue slots idle)
    saturation = None
    if rank == 0 and world == 1 and mode == "oqpsk10500" and not a.no_saturation and not a.channels:
        saturation = []
        pcm0, fcs0 = pipe.pcm, pipe.fcs
        for p in pipes:
            p.close()
        for Cs in (8192, 16384, 32768):
            try:
                ps = Pipeline(mode, Cs, 0, ebn0, envs_t, dev, local, stream)
                for _ in range(2):
                    ps.step_device()
                torch.cuda.synchronize()
                s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s0.record(stream)
                for _ in range(3):
                    ps.step_device()
                s1.record(stream)
                torch.cuda.synchronize()
                msx = s0.elapsed_time(s1) / 3
                v = Cs * STEP_SAMPLES / (msx * 1e-3) / 1e6
                saturation.append({"channels": Cs, "value": v, "unit": "Msamples/s", "channels_rt": v * 1e6 / FS, "ms_per_step": msx,
                                   "frac": (ALG_STEP * v * 1e6 / 1e9) / float(peaks.get("hbm_gbs", 6650.0))})
                ps.close(); del ps
                torch.cuda.empty_cache()
            except Exception as ex:                # e.g. out of memory on a smaller part
                saturation.append({"channels": Cs, "error": str(ex)[:120]})
                break
        pipe = None

    cpu_base = None
    if rank == 0 and not a.no_cpu_baseline:
        secs = max(1, int(round(a.cpu_seconds)))
        src = pipe.pcm if pipe is not None else pcm0
        fcsx = pipe.fcs if pipe is not None else fcs0
        rows = [src[i].cpu().numpy().copy() for i in range(cores)]
        jobs = [(m["kind"], m["fb"], m["lockingbw"], rows[i], secs, float(fcsx[i])) for i in range(cores)]
        cpu_base = cpu_baseline_block(jobs, cores, "%d channels x %d s of the same synthetic workload (the 1 s signal looped), one process per core, 100 ms writeData calls, demod + P-channel decode with DCD fed back" % (cores, secs))

    if rank == 0:
        line = {"metric": m["metric"], "value": value, "unit": "Msamples/s", "n_gpus": world,
                "steps": a.steps, "warmup": max(3, a.warmup), "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic", "channels_rt": value * 1e6 / FS,
                "config": {"workload": m["label"], "channels_per_gpu": C, "seconds_per_step": 1.0, "ebn0_db": ebn0,
                           "parallelism": "channels sharded x%d GPUs x %d concurrent batches per GPU, no data-path collective" % (world, G),
                           "l2": "inputs (%.0f MB int16 + %.1f GB of ring state per step) exceed the 126 MB L2" % (C * STEP_SAMPLES * 2 / 1e6, C * 3.4e-3)},
                "e2e": e2e, "gpu_launches": int(launches), "clocks": clk, "roofline": roofline, "cpu_baseline": cpu_base,
                "decode": {"su_total": tot[0], "su_crc_ok": tot[1], "channels_with_dcd": tot[2]}}
        if saturation is not None:
            line["saturation"] = saturation
        print(json.dumps(line))
    if pipe is not None:
        for p in pipes:
            p.close()
    if world > 1:
        import torch.distributed as dist
        dist.barrier(); dist.destroy_process_group()
    return 0


def run_burst(a):
    """BASELINE configs[3]: samples/1200bps_burst_sample1.wav (committed as tests/golden/burst_msk_1200_a_excerpt.npz, the whole
    521 155-sample recording) replicated over 2048 channels per GPU, replica r = Re{hilbert(x) e^(j 2 pi df_r n/Fs)},
    df_r = U(-300, 300) Hz from seed 0xB0057 + r; base PCM broadcast from rank 0 (ncclBroadcast); burst MSK demodulator (Hilbert
    FFT-FIR, burst detector, trident FFT acquisition, gated tail) + R/T packet layer. One step = one pass over the recording."""
    import torch
    from jaero_b200 import shard, synth
    import jaero_b200
    cores = usable_cores()
    base_np = np.load(os.path.join(ROOT, "tests", "golden", "burst_msk_1200_a_excerpt.npz"))["pcm"]
    metric = "IQ Msamples/s (1200 bps burst MSK demod + R/T packet decode)"
    label = "1200 bps burst MSK recording x2048 replicas with random frequency offsets, trident FFT acquisition + R/T packets (BASELINE configs[3])"
    if a.impl == "reference":
        if int(os.environ.get("RANK", "0")) != 0:
            return 0
        reps = synth.offset_replicas(base_np, synth.replica_offsets(0, cores))
        jobs = [("burst_msk", 1200, 1800, reps[i], 1, 1000.0) for i in range(cores)]
        cpu_reference_run(jobs[:1], 1)
        impl, samples, busy, wall, tot, ok = cpu_reference_run(jobs, cores)
        val = samples / busy / 1e6
        print(json.dumps({"impl": "reference", "metric": metric, "value": val, "unit": "Msamples/s", "n_gpus": max(a.gpus, int(os.environ.get("WORLD_SIZE", "1"))),
                          "steps": 1, "warmup": 1, "ms_per_step": busy * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                          "dtype": "f64", "data": "recording replicas", "config": {"workload": label + "; reference arm = %d replicas" % cores},
                          "cpu_baseline": {"value": val, "unit": "Msamples/s", "cores": cores, "kind": impl, "sample": "%d replicas x 10.86 s" % cores},
                          "e2e": {"value": val, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                          "decode": {"t_packets": tot}, "gpu_launches": 0}))
        return 0
    rank, local, world = shard.init_from_env()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    C = a.channels or 2048
    base = torch.zeros(len(base_np), dtype=torch.int16, device=dev)
    if rank == 0:
        base.copy_(torch.from_numpy(base_np))
    shard.broadcast_(base.view(torch.uint8), 0)     # (NCCL has no int16: the same bytes as uint8) the one collective of this workload: the shared recording over NCCL/NVLink
    offs = synth.replica_offsets(rank * C, rank * C + C)
    n = len(base_np)
    pitch = (n + 7) & ~7
    pcm = torch.zeros((C, pitch), dtype=torch.int16, device=dev)
    pcm[:, :n] = offset_replicas_gpu(base, offs, dev)
    torch.cuda.synchronize()
    chunk = 49152

    def one_pass(host=None, read=False):
        b = jaero_b200.BurstMskBatch(C, fb=1200.0, freq_center=1000.0, lockingbw=1800.0, signalthreshold=0.6, device=local)
        rt = jaero_b200.RTChannelBatch(C, 1200, device=local)
        npk = 0
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for s0 in range(0, n, chunk):
            m = min(chunk, n - s0)
            if host is None:
                b.write_device(pcm.data_ptr() + 2 * s0, m, pitch)
            else:
                b.write(host[:, s0:s0 + m])
            rt.process_burst(b)
            if read:
                npk += sum(len(p) for p in rt.read_packets())
        b.sync(); torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        st = b.status()
        launches = b.launches + rt.launches
        tr, bad, dcd = rt.stats()
        b.close(); rt.close()
        return dt, launches, int(sum(s["n_sig_true"] for s in st)), npk, int(tr.sum())

    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    one_pass()                                       # warm-up pass (module load, allocations); W further passes below
    for _ in range(max(0, min(a.warmup, 3) - 1)):
        one_pass()
    shard.barrier()
    clocks.mark_begin()
    dts, launches, bursts = [], 0, 0
    for _ in range(a.steps):
        dt, l, nb, _, trials = one_pass()
        dts.append(dt); launches += l; bursts = nb
    ms = shard.reduce_max(sum(dts) * 1e3, device=dev)
    clk = clocks.stop() if rank == 0 else None
    total = float(C) * n * a.steps * world
    value = total / (ms * 1e-3) / 1e6
    e2e = None
    if not a.no_e2e:
        host = pcm[:, :n].cpu().numpy()
        dt, _, _, npk, _ = one_pass(host=host, read=True)
        ems = shard.reduce_max(dt * 1e3, device=dev)
        e2e = {"value": float(C) * n * world / (ems * 1e-3) / 1e6, "unit": "Msamples/s", "h2d_bytes_per_step": int(C * n * 2), "d2h_bytes_per_step": int(C * 8 * 160),
               "ms_per_step": ems, "t_packets": npk}
    allb = shard.reduce_sum([float(bursts)], device=dev)
    cpu_base = None
    if rank == 0 and not a.no_cpu_baseline:
        reps = pcm[:cores, :n].cpu().numpy()
        jobs = [("burst_msk", 1200, 1800, reps[i].copy(), 1, 1000.0) for i in range(cores)]
        cpu_base = cpu_baseline_block(jobs, cores, "%d replicas x 10.86 s, one process per core, burst demod + R/T packet decode" % cores)
    if rank == 0:
        print(json.dumps({"metric": metric, "value": value, "unit": "Msamples/s", "n_gpus": world, "steps": a.steps, "warmup": max(1, min(a.warmup, 3)),
                          "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
                          "data": "recording replicas (Hilbert-rotated, seeds 0xB0057 + r)", "channels_rt": value * 1e6 / FS,
                          "config": {"workload": label, "channels_per_gpu": C, "samples_per_step": n,
                                     "timing": "host clock around device synchronize: the burst path synchronises once per 16384-sample chunk to size its trident FFT launches",
                                     "collective": "ncclBroadcast of the base PCM (%d bytes) from rank 0" % (2 * n)},
                          "e2e": e2e, "gpu_launches": int(launches), "clocks": clk, "cpu_baseline": cpu_base,
                          "decode": {"bursts_acquired": allb[0]}}))
    if world > 1:
        import torch.distributed as dist
        dist.barrier(); dist.destroy_process_group()
    return 0


def run_mix(a):
    """BASELINE configs[4]: 12 288 x 10.5 kbps OQPSK P-channels + 4096 x 8400 bps C-channels (3:1), contiguous cost-weighted
    shards (jaero_b200.shard.weighted_ranges), no data-path collective. --scaling weak: 2048 channels per GPU (the mix scaled
    down); strong: the 16 384-channel set split over the GPUs. The 8400 bps signal is the reference's own C-channel recording
    (tests/golden/oqpsk_8400_excerpt.npz, 8 s) given a per-channel frequency offset (Hilbert rotation) - real frames, real SUs."""
    import torch
    from jaero_b200 import shard, synth
    import jaero_b200
    rank, local, world = shard.init_from_env()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    total_ch = 16384 if a.scaling == "strong" else 2048 * world
    if a.channels:
        total_ch = a.channels * (world if a.scaling == "weak" else 1)
    n_c = total_ch // 4                                            # 8400 bps share
    n_p = total_ch - n_c
    COST_8400 = 3.0                                                # measured relative cost per channel (single-warp K1a' + K6), see DESIGN.md
    costs = [1.0] * n_p + [COST_8400] * n_c
    lo, hi = shard.weighted_ranges(costs, world)[rank]
    p_lo, p_hi = min(lo, n_p), min(hi, n_p)
    c_lo, c_hi = max(lo, n_p) - n_p, max(hi, n_p) - n_p
    cp, cc = p_hi - p_lo, c_hi - c_lo
    envs_t = torch.zeros((16, STEP_SAMPLES), dtype=torch.complex64, device=dev)
    if rank == 0:
        envs_t.copy_(torch.from_numpy(base_envelopes("oqpsk10500", 16, 7)))
    shard.broadcast_(torch.view_as_real(envs_t), 0)
    base8 = np.load(os.path.join(ROOT, "tests", "golden", "oqpsk_8400_excerpt.npz"))["pcm"]
    b8 = torch.zeros(len(base8), dtype=torch.int16, device=dev)
    if rank == 0:
        b8.copy_(torch.from_numpy(base8))
    shard.broadcast_(b8.view(torch.uint8), 0)       # NCCL has no int16 type: the same bytes as uint8
    sA, sB = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    pipe = Pipeline("oqpsk10500", cp, p_lo, 10.0, envs_t, dev, local, sA) if cp > 0 else None
    cb = cl = pcm8 = None
    n8 = (len(base8) // STEP_SAMPLES) * STEP_SAMPLES
    if cc > 0:
        offs = synth.replica_offsets(n_p + c_lo, n_p + c_hi, span_hz=200.0, seed0=0xC8400)
        pcm8 = offset_replicas_gpu(b8[:n8], offs, dev)
        cb = jaero_b200.DemodBatch("oqpsk", cc, fb=8400, freq_center=8000.0, lockingbw=10500, afc=True, device=local)
        cl = jaero_b200.CChannelBatch(cc, device=local)
        cb.set_stream(sB.cuda_stream)
    k8 = [0]

    def step():
        if pipe is not None:
            pipe.step_device()
        if cb is not None:
            s0 = (k8[0] % (n8 // STEP_SAMPLES)) * STEP_SAMPLES; k8[0] += 1
            cb.write_device(pcm8.data_ptr() + 2 * s0, STEP_SAMPLES, pcm8.stride(0))
            cl.process_batch(cb)
            cl.tick(cb)
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    for _ in range(max(3, a.warmup)):
        step()
    torch.cuda.synchronize(); shard.barrier()
    l0 = (pipe.launches if pipe else 0) + (cb.launches + cl.launches if cb else 0)
    e0, e1, eB = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True), torch.cuda.Event()
    clocks.mark_begin()
    e0.record(sA)
    sB.wait_event(e0)                                             # neither stream starts before e0 ...
    for _ in range(a.steps):
        step()
    eB.record(sB); sA.wait_event(eB)                              # ... and e1 fires when both are done
    e1.record(sA)
    torch.cuda.synchronize(); shard.barrier()
    ms = shard.reduce_max(e0.elapsed_time(e1), device=dev)
    launches = (pipe.launches if pipe else 0) + (cb.launches + cl.launches if cb else 0) - l0
    clk = clocks.stop() if rank == 0 else None
    value = float(total_ch) * STEP_SAMPLES * a.steps / (ms * 1e-3) / 1e6
    okp = float(pipe.layer.stats()[2].sum()) if pipe else 0.0
    okc = float(cl.stats()[2].sum()) if cl else 0.0
    if cl is not None:
        cl.read_frames()                                          # drain (also checks the frame queue did not overflow)
    tot = shard.reduce_sum([okp, okc, float(cp), float(cc)], device=dev)
    if rank == 0:
        print(json.dumps({"metric": "IQ Msamples/s (10.5k OQPSK + 8400 bps C-channel mix, demod + Viterbi)", "value": value, "unit": "Msamples/s",
                          "n_gpus": world, "steps": a.steps, "warmup": max(3, a.warmup), "ms_per_step": ms / a.steps, "higher_is_better": True,
                          "scaling": a.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic 10.5k + recording replicas 8400", "channels_rt": value * 1e6 / FS,
                          "config": {"workload": "10.5 kbps OQPSK P-channels + 8400 bps C-channels 3:1 (BASELINE configs[4])", "channels_total": total_ch,
                                     "p_channels": n_p, "c_channels": n_c, "cost_weight_8400": COST_8400,
                                     "parallelism": "contiguous cost-weighted channel ranges x%d, no data-path collective; the two modes of a rank run on two streams" % world},
                          "gpu_launches": int(launches), "clocks": clk, "e2e": None, "cpu_baseline": None,
                          "decode": {"p_su_crc_ok": tot[0], "c_su_crc_ok": tot[1], "p_channels_sum": tot[2], "c_channels_sum": tot[3]}}))
    if pipe is not None:
        pipe.close()
    if cb is not None:
        cb.close(); cl.close()
    if world > 1:
        import torch.distributed as dist
        dist.barrier(); dist.destroy_process_group()
    return 0


def main():
    a = parse()
    if a.workload in MODES:
        return run_continuous(a, a.workload)
    if a.workload == "burst1200x2048":
        return run_burst(a)
    if a.impl == "reference":
        if int(os.environ.get("RANK", "0")) == 0:
            print(json.dumps({"impl": "reference", "unavailable": "mix16384 has no separate reference arm: see the oqpsk10500 arm (its 10.5k share) and tools/cpu_modes.py"}))
        return 0
    return run_mix(a)


if __name__ == "__main__":
    sys.exit(main())
