"""Device channelizer measurement. One JSON line per configuration on stdout (and appended to --out if given).

A  channelizer alone: cs16 IQ at --input-rate (default 2.4 MHz) resident on the device (seeded noise), C = 192 and 4096
   channels. 1 s of IQ warm-up, then three timed repeats of 10 s of IQ each (1 s per write), CUDA events on the handle's
   stream. Reports ms per second of IQ, the real-time factor, FP32 FLOP/s achieved from 8*Tp*C*M_out (Tp taps per polyphase
   branch, M_out outputs; Tp = T at integer rates), output bytes, and a per-kernel breakdown taken with torch.profiler in a
   separate pass. Rates that are not a multiple of 48 kHz (2.048 MHz: L/M = 3/128) run the polyphase path.
B  end to end, 4096 channels of OQPSK 10.5k: IQ at --input-rate carrying 64 distinct carriers, 64 channels tuned to each. Per 1 s
   step, on one stream: channelizer -> DemodBatch.write_device -> PChannelBatch.process_batch. Alternates, in the same
   process, with the same step fed device-resident PCM (a captured second of the channelizer's output), and with both
   inputs coming from pinned host memory (IQ through Channelizer.write, PCM through DemodBatch.write).

python tools/chan_bench.py [--configs A,B] [--input-rate HZ] [--out FILE]   (needs a CUDA device; there is no CPU path)
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import jaero_b200 as jb  # noqa: E402
from jaero_b200 import synth  # noqa: E402

FO, AUDIO = 48000.0, 12000.0
FS = 2.4e6                                                  # --input-rate


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.sm", "--format=csv"], capture_output=True, text=True)
    return dict(device=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip().splitlines()[-1] if q.returncode == 0 else q.stderr.strip())


def stats(v):
    v = sorted(v)
    return dict(median=v[len(v) // 2], min=v[0], max=v[-1], spread_pct=100.0 * (v[-1] - v[0]) / v[len(v) // 2])


def emit(rec, out):
    line = json.dumps(rec, sort_keys=True)
    print(line, flush=True)
    if out:
        with open(out, "a") as fh:
            fh.write(line + "\n")


def config_a(C, info, out, secs=10, repeats=3):
    g = torch.Generator(device="cuda").manual_seed(1234 + C)
    n1 = int(FS)
    iq = torch.randint(-3000, 3000, (secs * n1, 2), dtype=torch.int16, device="cuda", generator=g)
    edge = FS / 2 - 6000.0
    off = np.linspace(-edge, edge - 1.0, C) + 0.37          # off the 1 Hz grid, inside the band
    s = torch.cuda.Stream()
    ch = jb.Channelizer(off, FS, output_rate=FO, audio_hz=AUDIO, passband_hz=12000.0)
    ch.set_stream(s.cuda_stream)
    T = len(jb.channelizer_taps(FS, output_rate=FO, audio_hz=AUDIO, passband_hz=12000.0))
    L, Mr = jb.channelizer_ratio(FS, output_rate=FO, audio_hz=AUDIO, passband_hz=12000.0)
    Tp = (T + L - 1) // L
    torch.cuda.synchronize()
    ch.write_device(iq.data_ptr(), n1)                      # warm-up: 1 s of IQ
    ch.sync()
    times = []
    for _ in range(repeats):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(s)
        for k in range(secs):
            ch.write_device(iq.data_ptr() + k * n1 * 4, n1)
        e1.record(s)
        e1.synchronize()
        times.append(e0.elapsed_time(e1) / secs)
    M = n1 * L // Mr                                        # outputs per second of IQ
    st = stats(times)
    flop = 8.0 * Tp * C * M
    # per-kernel breakdown, profiler pass of its own (2 s of IQ)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for k in range(2):
            ch.write_device(iq.data_ptr() + k * n1 * 4, n1)
        ch.sync()
    kern = {}
    for e in prof.key_averages():
        if "chan_" in e.key:
            name = "chan_ddc_kernel" if "ddc" in e.key else "chan_convert_kernel"
            kern[name] = round(e.device_time_total / 1000.0 / 2, 3)   # ms per second of IQ
    rec = dict(config="A", channels=C, input_rate=FS, output_rate=FO, taps=T, ratio=[L, Mr], taps_per_phase=Tp, iq_format="cs16", secs_per_repeat=secs,
               ms_per_s_iq=st, realtime_factor=1000.0 / st["median"], fp32_tflops=flop / (st["median"] * 1e-3) / 1e12,
               flop_per_s_iq=flop, output_bytes_per_s_iq=C * M * 2, input_bytes_per_s_iq=n1 * 4,
               kernel_ms_per_s_iq=kern, launches_per_write=2, **info)
    emit(rec, out)
    ch.close()


def _pchan_env(seed, n_frames=2):
    bits, _ = synth.pchannel_bits(10500, n_frames, seed, return_sus=True, loop=True)
    return synth.oqpsk_envelope(bits, 10500)


def config_b(info, out, steps=10, repeats=3, n_car=64, per=64):
    C = n_car * per
    car_off = np.array([-1.1e6 + 35000.0 * k + 1000.0 + 7 * k for k in range(n_car)])   # whole hertz: the 1 s loop stays seamless
    iq1 = synth.wideband_iq([_pchan_env(500 + k) for k in range(n_car)], car_off, FS, amplitudes=np.full(n_car, 300.0),
                            ebn0_db=10.0, fb=10500.0, seed=77)
    off = np.repeat(car_off, per)
    n1 = len(iq1)
    assert n1 == int(FS)
    d_iq = torch.from_numpy(iq1).cuda()
    h_iq = torch.from_numpy(iq1).pin_memory()
    s = torch.cuda.Stream()

    def chain(with_chan):
        ch = jb.Channelizer(off, FS, output_rate=FO, audio_hz=AUDIO, passband_hz=12000.0) if with_chan else None
        b = jb.DemodBatch("oqpsk", C, fb=10500, freq_center=AUDIO)
        pc = jb.PChannelBatch(C, 10500)
        for o in (ch, b):
            if o is not None:
                o.set_stream(s.cuda_stream)
        return dict(ch=ch, b=b, pc=pc)

    # a captured second of the channelizer's output is the PCM the PCM-fed chains see
    cap = chain(True)
    cap["ch"].write_device(d_iq.data_ptr(), n1)
    cap["ch"].write_device(d_iq.data_ptr(), n1)
    pcm = torch.from_numpy(cap["ch"].read()).cuda()
    h_pcm = torch.from_numpy(pcm.cpu().numpy()).pin_memory()
    for o in cap.values():
        o.close()
    variants = dict(iq_device=chain(True), pcm_device=chain(False), iq_host=chain(True), pcm_host=chain(False))
    h_pcm_np = h_pcm.numpy()

    def step(name, v):
        if name == "iq_device":
            v["ch"].write_device(d_iq.data_ptr(), n1)
        elif name == "iq_host":
            v["ch"].write(h_iq.numpy())
        if v["ch"] is not None:
            p, n, st = v["ch"].output_device()
            v["b"].write_device(p, n, st)
        elif name == "pcm_device":
            v["b"].write_device(pcm.data_ptr(), pcm.shape[1], pcm.shape[1])
        else:
            v["b"].write(h_pcm_np)
        v["pc"].process_batch(v["b"])
        v["pc"].discard_sus()

    torch.cuda.synchronize()
    for name, v in variants.items():                        # warm-up: 1 s each
        step(name, v)
    torch.cuda.synchronize()
    times = {k: [] for k in variants}
    for _ in range(repeats):
        for name, v in variants.items():                    # alternate the variants inside each repeat
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            e0.record(s)
            for _k in range(steps):
                step(name, v)
            e1.record(s)
            e1.synchronize()
            times[name].append(dict(ev=e0.elapsed_time(e1) / steps, wall=(time.perf_counter() - t0) * 1000.0 / steps))
    res = {}
    for name, v in variants.items():
        dcd, tot, ok = v["pc"].stats()
        res[name] = dict(ms_per_step=stats([t["wall"] for t in times[name]]), event_ms_per_step=stats([t["ev"] for t in times[name]]),
                         dcd_channels=int(dcd.sum()), su_total=int(tot.sum()), su_crc_ok=int(ok.sum()))
    rec = dict(config="B", channels=C, distinct_carriers=n_car, input_rate=FS, steps_per_repeat=steps, step_s=1.0,
               chan_added_ms_per_step=res["iq_device"]["ms_per_step"]["median"] - res["pcm_device"]["ms_per_step"]["median"],
               h2d_bytes_per_step=dict(iq=n1 * 4, pcm=int(pcm.numel()) * 2), variants=res, **info)
    emit(rec, out)
    for v in variants.values():
        for o in v.values():
            if o is not None:
                o.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="A,B")
    ap.add_argument("--out", default=None)
    ap.add_argument("--secs", type=int, default=10)
    ap.add_argument("--input-rate", type=float, default=2.4e6)
    a = ap.parse_args()
    global FS
    FS = a.input_rate
    if not torch.cuda.is_available() or jb.lib().jaero_device_count() < 1:
        sys.exit("chan_bench: needs a CUDA device (there is no CPU path)")
    info = device_info()
    cfg = a.configs.split(",")
    if "A" in cfg:
        for C in (192, 4096):
            config_a(C, info, a.out, secs=a.secs)
    if "B" in cfg:
        config_b(info, a.out, steps=a.secs)


if __name__ == "__main__":
    main()
