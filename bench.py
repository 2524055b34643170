#!/usr/bin/env python
"""bench.py — NRSC-5 FM receive-chain throughput on B200 (see DESIGN.md §measurement).

Metric (BASELINE.json): cu8 I/Q Msamples/s (complex samples; / 1.488375 = x real
time) of the whole hot path, at N GPUs, streams sharded per GPU, weak scaling.

A *step* = one pass of the hot path over one batch: S independent synthetic
FM MP1 channels per GPU (config 5's per-GPU shard: 128 channels), each
`frames` L1 frames (+2 blocks of tail) long, decoded from reset to L1 PDUs.

  value : whole-job Msamples/s with the cu8 already resident in HBM when the
          timed region starts (engine attached to a device buffer).
  e2e   : same metric through the public C ABI with HOST buffers: pinned
          host->device copy of every stream's cu8 and device->host drain of all
          PDU/event records inside the timed region (and, for N>1, an NCCL
          gather of the fixed-size P1 PDU slabs to rank 0).
  --impl reference : the reference's own CPU implementation (the UNMODIFIED
          reference built into oracle/_ref/libnrsc5_ref.so; FFTW replaced by
          oracle/shim/fftshim.c) on the host cores, same captures.

One JSON line on stdout (rank 0).
"""
from __future__ import annotations

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

SAMPLE_RATE = 1488375.0
BLOCK_BYTES = 276480
DEMOD_BYTES_PER_BLOCK = 276480 + 32 * 534 * 8      # cu8 in + 534 complex bins x 32 symbols out (DESIGN.md)
FUSED_BYTES_PER_BLOCK = 276480 + 23040              # SURVEY §8(d): cu8 in + int8 soft bits out
P1_BYTES_PER_FRAME = 368640 + 18272 + 160           # SURVEY §8(d)
SYNC_BYTES_PER_BLOCK = 32 * 534 * 8 + 23040


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--streams", type=int, default=128, help="channels per GPU")
    ap.add_argument("--frames", type=int, default=4, help="L1 frames per channel per step (SURVEY §8d config 5: 4)")
    ap.add_argument("--distinct", type=int, default=4, help="distinct synthetic captures (replicated with offsets)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dbg", type=int, default=0, help="kernel experiment switches (nrsc5b_debug_set)")
    ap.add_argument("--no-l2", action="store_true", help="skip the L2-on-device leg (SURVEY 8 f1)")
    ap.add_argument("--l2-leg", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--no-am", action="store_true", help="skip the AM leg (BASELINE config 4)")
    ap.add_argument("--am-leg", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--no-mp3", action="store_true", help="skip the MP3 leg (BASELINE config 3)")
    ap.add_argument("--mp3-leg", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--no-chan", action="store_true", help="skip the channeliser leg (SURVEY 8 f3)")
    ap.add_argument("--chan-leg", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--no-dropin", action="store_true", help="skip the single-stream drop-in leg (BASELINE configs 1, 2)")
    ap.add_argument("--dropin-leg", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--mp3-streams", type=int, default=64)
    ap.add_argument("--mp3-frames", type=int, default=6)
    ap.add_argument("--am-streams", type=int, default=256)
    ap.add_argument("--am-frames", type=int, default=12)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the records of the last timed step as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def make_captures(distinct: int, frames: int, base_seed: int = 1234):
    from nrsc5_b200 import synth
    caps = []
    for i in range(distinct):
        kw = dict(nframes=frames, seed=base_seed + i, lead_in=0, tail_blocks=2, noise_seed=5 + i)
        if i % 4 == 1:
            kw.update(cfo_hz=120.0)
        elif i % 4 == 2:
            kw.update(cfo_hz=-300.0, noise_lsb=12.0)
        elif i % 4 == 3:
            kw.update(cfo_hz=60.0, noise_lsb=6.0)
        caps.append(synth.make_fm_mp1(**kw).cu8)
    return caps


def make_l2_captures(distinct: int, frames: int, base_seed: int = 4321):
    """Captures whose P1 PDUs carry real L2 content (audio PDUs with ~45 packets, PSD, header expansion fields,
    correctable header errors: nrsc5_b200/synth_l2.py); the first L1 frame keeps the plain PDU."""
    from nrsc5_b200 import synth, synth_l2
    caps, packets = [], []
    for i in range(distinct):
        fr = [f for f in synth_l2.make_l2_sequence(seed=base_seed + i, nframes=max(1, frames - 1)) if f is not None]
        cap = synth.make_fm_mp1(nframes=frames, seed=base_seed + i, lead_in=0, tail_blocks=2, noise_seed=5 + i,
                                cfo_hz=(0.0, 120.0)[i % 2], p1_frames=[None] + [f[2] for f in fr])
        caps.append(cap.cu8)
    return caps


def l2_leg(args):
    """The same job with L2 framing on the device (nrsc5b_enable_l2): every decoded frame also goes through k_l2 and
    leaves as a REC_L2 record (HDC packets with CRC verdicts, PSD messages, service changes).  Run by the main bench
    in a subprocess (rank 0, N=1) so that this newer kernel cannot disturb the headline measurement; prints one JSON
    object."""
    import torch
    import nrsc5_b200
    from nrsc5_b200 import engine as eng
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    S = args.streams
    caps = make_l2_captures(2, args.frames)
    views, nbytes = stream_views(caps, S, 0)
    host = torch.empty((S, nbytes), dtype=torch.uint8).pin_memory()
    hnp = host.numpy()
    for s, v in enumerate(views):
        hnp[s, :] = v
    devbuf = torch.empty((S, nbytes + 64), dtype=torch.uint8, device=dev)
    devbuf[:, :nbytes].copy_(host)
    devbuf[:, nbytes:] = 127
    torch.cuda.synchronize()
    stream = torch.cuda.current_stream()
    log_cap = (args.frames + 1) * (18272 + 64 + 18272 + 16384) + 96 * 1024
    e = nrsc5_b200.Engine(nstreams=S, input_capacity=nbytes + 4096, device=0, log_capacity=log_cap)
    e.set_cuda_stream(stream.cuda_stream)

    def step(l2):
        e.enable_l2(l2)
        e.attach_device_input(devbuf.data_ptr(), nbytes + 64, nbytes)
        e.rewind()
        e.process()

    def timed(l2, steps):
        for _ in range(3):
            step(l2)
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        for _ in range(steps):
            step(l2)
        ev1.record(stream)
        torch.cuda.synchronize()
        return ev0.elapsed_time(ev1) / steps

    # gate: the packets the generator put into stream 0's PDUs come out, with intact CRCs
    step(True)
    recs = e.drain(0)
    l2 = [r for t, r in recs if t == eng.REC_L2]
    pk = [ev for r in l2 for t, ev in r["events"] if t == eng.EV_PACKET]
    assert len(l2) >= 2 and len(pk) >= 30 * (len(l2) - 1), (len(l2), len(pk))
    assert all(p["flags"] == 0 for p in pk) and not any(r["flags"] for r in l2)
    steps = args.steps
    ms_off = timed(False, steps)
    ms_on = timed(True, steps)
    e.set_profiling(True)
    step(True)
    torch.cuda.synchronize()
    kt = e.kernel_times()
    e.set_profiling(False)
    frames_per_step = int(e.stats().p1_frames)
    samples = S * (nbytes // 2)
    k = kt.get("l2", {"ms": 0.0, "launches": 0})
    # algorithmic bytes of k_l2 per frame: 18 272 B of packed frame bits in, 18 269 B of PDU + the event list out
    ev_bytes = sum(8 + 28 for _ in pk) / max(1, len(l2))
    alg = frames_per_step * (18272 + 18272 + 40 + ev_bytes)
    peak, _ = measured_peak()
    out = {"value": samples / (ms_on * 1e-3) / 1e6, "unit": "Msamples/s", "ms_per_step": ms_on,
           "same_workload_l1_only": {"value": samples / (ms_off * 1e-3) / 1e6, "ms_per_step": ms_off},
           "k_l2": {"ms_per_step": k["ms"], "launches": k["launches"], "frames_per_step": frames_per_step,
                    "alg_bytes_per_step": alg, "achieved_gbs": (alg / (k["ms"] * 1e-3) / 1e9) if k["ms"] > 0 else 0.0,
                    "peak_gbs": peak, "note": "one CTA per stream; the PDU walk is sequential per frame (thread 0), "
                                              "PCI strip / CRC-8 / record copy use the whole CTA"},
           "packets_per_frame": len(pk) / max(1, len(l2) - 1), "steps": steps,
           "workload": f"{S} synthetic FM MP1 channels x {args.frames} L1 frames, P1 PDUs with real audio PDUs "
                       "(synth_l2.py), cu8 resident in HBM, L2 framing on the device (REC_L2 per frame)"}
    print(json.dumps(out), flush=True)
    e.close()


def mp3_leg(args):
    """BASELINE config 3: `--mp3-streams` synthetic FM MP3 (extended hybrid) channels, `--mp3-frames` L1 frames each,
    batched on one GPU: P1, PIDS and the P3 frames of the PX1 partitions (interleaver IV) decoded from reset.
    `value`: samples resident in HBM (nrsc5b_rewind -> process); `e2e`: reset -> push -> process -> drain.  Host
    clock around synchronous calls.  Run by the main bench in a subprocess (rank 0, N=1); prints one JSON object."""
    import nrsc5_b200
    from nrsc5_b200 import engine as eng, synth
    S, F = args.mp3_streams, args.mp3_frames
    caps = [synth.make_fm_mp3(nframes=F, seed=11 + i, lead_in=0, tail_blocks=2, cfo_hz=(0.0, 80.0)[i % 2]).cu8 for i in range(2)]
    views, nbytes = stream_views(caps, S, 0)
    views = [np.ascontiguousarray(v) for v in views]
    log_cap = (F + 1) * (18272 + 64) + 8 * F * (576 + 32) + 128 * 1024
    e = nrsc5_b200.Engine(nstreams=S, input_capacity=nbytes + 4096, log_capacity=log_cap)

    def step():
        t0 = time.perf_counter()
        e.reset()
        for s in range(S):
            e.push_cu8(s, views[s])
        e.process()
        recs = e.drain_all()
        return time.perf_counter() - t0, recs

    _, recs = step()
    gate = parity_gate(views, recs, what="mp3_config3")           # every channel: P1 / PIDS / P3 PDUs in order == oracle
    nf = [(sum(1 for t, r in rr if t == eng.REC_FRAME and r["lc"] == 0), sum(1 for t, r in rr if t == eng.REC_FRAME and r["lc"] == 1))
          for rr in recs]
    assert nf[0][0] >= F - 1 and nf[0][1] >= 8 * (F - 2) - 2, nf[0]         # P3 output starts after two frames of interleaver fill
    first = [record_digest(r) for r in recs]
    steps = args.steps
    tot = sum(step()[0] for _ in range(steps))
    res = 0.0
    for _ in range(steps):
        e.rewind()
        t0 = time.perf_counter()
        e.process()
        res += time.perf_counter() - t0
    again = e.drain_all()
    assert [record_digest(r) for r in again] == first, "rewind -> process gave other records than reset -> push -> process"
    samples = S * (nbytes // 2)
    out = {"value": samples * steps / res / 1e6, "unit": "Msamples/s", "x_realtime": samples * steps / res / SAMPLE_RATE,
           "ms_per_step": 1e3 * res / steps,
           "e2e": {"value": samples * steps / tot / 1e6, "ms_per_step": 1e3 * tot / steps, "x_realtime": samples * steps / tot / SAMPLE_RATE,
                   "h2d_bytes_per_step": int(S * nbytes), "what": "reset -> nrsc5b_push_cu8 per channel from host memory -> process -> drain_all"},
           "steps": steps, "timing": "host clock around synchronous calls (the engine waits for its kernels)",
           "p1_frames_per_channel": nf[0][0], "p3_frames_per_channel": nf[0][1], "parity_gate": gate,
           "workload": f"{S} synthetic FM MP3 channels x {F} L1 frames (+2 blocks), cu8, full chain to P1 / PIDS / P3 PDUs"}
    print(json.dumps(out), flush=True)
    e.close()


def am_leg(args, engine_factory=None):
    """BASELINE config 4: `--am-streams` synthetic AM MA1 channels (cs16 at 46 511.72 S/s, `--am-frames` L1 frames
    each) on one GPU, decoded from reset to L1 PDUs by the AM engine (one warp per stream, first unoptimised path).
    A step = reset, push every channel's samples from host memory (nrsc5b_push_cs16), process, drain: the whole
    thing is timed on the host clock around synchronous calls (the engine waits for its own kernels), and the
    process() part alone is reported next to it.  Run by the main bench in a subprocess (rank 0, N=1); prints one
    JSON object."""
    import nrsc5_b200
    from nrsc5_b200 import engine as eng, synth_am
    S, F = args.am_streams, args.am_frames
    caps = [synth_am.make_am_ma1(nframes=F, seed=3 + i, lead_in=500 + 64 * i, cfo_hz=(0.0, 1.5)[i % 2]).cs16 for i in range(2)]
    n = min(c.size for c in caps) - 2 * 512
    views = [np.ascontiguousarray(caps[s % 2][2 * ((37 * (s // 2)) % 256):][:n]) for s in range(S)]
    make = engine_factory or (lambda **kw: nrsc5_b200.Engine(**kw))
    e = make(nstreams=S, input_capacity=2 * n + 4096, log_capacity=512 << 10, mode="am")

    def step():
        t0 = time.perf_counter()
        e.reset()
        for s in range(S):
            e.push_cs16(s, views[s])
        t1 = time.perf_counter()
        e.process()
        t2 = time.perf_counter()
        recs = e.drain_all()
        t3 = time.perf_counter()
        return t3 - t0, t2 - t1, recs

    _, _, recs = step()                                   # warm-up + gate
    p1 = [r for t, r in recs[0] if t == eng.REC_FRAME and r["lc"] == 0]
    assert len(p1) >= 8 * (F - 8), f"{len(p1)} AM P1 frames decoded from {F} transmitted L1 frames"
    gate = parity_gate(views, recs, am=True, what="am_config4")   # every channel: P1 / P3 / PIDS PDUs in order == oracle
    first = [record_digest(r) for r in recs]
    steps = args.steps
    tot = proc = 0.0
    for _ in range(steps):
        a, b, _ = step()
        tot += a
        proc += b
    # the same samples again, already resident in HBM: rewind (receiver state starts over) + process
    res = 0.0
    for _ in range(steps):
        e.rewind()
        t0 = time.perf_counter()
        e.process()
        res += time.perf_counter() - t0
    again = e.drain_all()
    assert [record_digest(r) for r in again] == first, "rewind -> process gave other records than reset -> push -> process"
    samples = S * (n // 2)
    try:
        pc = e.am_phase_cycles()                          # of the last rewind -> process
        nblk = max(1, int(e.stats().blocks))
        am_phases = {k: round(v / nblk / 1965.0, 2) for k, v in pc.items() if k != "traceback_repair_rounds"}    # us per stream-block at 1965 MHz
        am_phases["traceback_repair_rounds_per_block"] = round(pc.get("traceback_repair_rounds", 0) / nblk, 4)   # (a count, not a time)
    except Exception:                                     # noqa: BLE001
        am_phases = None
    # the unmodified reference on this host's cores: one process per channel (cs16, AM mode), 3 passes each
    cpu = None
    try:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import reftap
        if reftap.available():
            v, nproc, info = cpu_reference_numbers(views, 2 * n, 3, am=True)     # (2 * n bytes // 2 = n int16 = n / 2 samples x 2)
            # cpu_reference_numbers counts nbytes // 2 units per pass: for cs16 that is int16 values; complex samples = half
            cpu = dict({"value": v / 2, "unit": "Msamples/s (cs16 complex)", "cores": nproc, "kind": "reference",
                        "sample": f"{nproc} processes x 3 passes over one {n // 2}-sample AM channel each"}, **info)
            cpu["single_core_value"] /= 2
            cpu["all_cores_value"] /= 2
    except Exception as ex:                                   # noqa: BLE001
        cpu = {"error": repr(ex)[:300]}
    peak, peak_src = measured_peak()
    blocks = int(e.stats().blocks)
    alg = 35640.0 * (samples / (8640.0))                      # SURVEY 8(d): 35 640 B of cs16 in per AM block (8 910 samples window, 8 640 new)
    ms = 1e3 * res / steps
    out = {"value": samples * steps / res / 1e6, "unit": "Msamples/s (cs16 complex, 46 511.72 S/s per channel)",
           "roofline": {"bound": "hbm", "kernel": "k_am (whole AM chain, one CTA per stream)", "achieved": alg / (ms * 1e-3) / 1e9, "peak": peak,
                        "unit": "GB/s", "frac": alg / (ms * 1e-3) / 1e9 / peak, "peak_source": peak_src, "traffic": None,
                        "note": "latency-bound by construction: per stream the NCO phase chain (17 280 dependent complex multiplications "
                                "per block, one warp) and the K=9 recursion (a verified chunk per warp, three trellis steps per metric "
                                "exchange) are dependent chains; 256 streams put at most two CTAs on an SM", "blocks_total": blocks},
           "cpu_baseline": cpu, "phases_us_per_stream_block_at_1965MHz": am_phases,
           "x_realtime": samples * steps / res / 46511.71875, "ms_per_step": 1e3 * res / steps,
           "e2e": {"value": samples * steps / tot / 1e6, "ms_per_step": 1e3 * tot / steps, "x_realtime": samples * steps / tot / 46511.71875,
                   "process_ms_per_step": 1e3 * proc / steps, "h2d_bytes_per_step": int(S * n * 2),
                   "what": "reset -> nrsc5b_push_cs16 per channel from host memory -> process -> drain_all"},
           "steps": steps, "timing": "host clock around synchronous calls (the engine waits for its kernels)",
           "p1_frames_per_channel": len(p1), "parity_gate": gate,
           "workload": f"{S} synthetic AM MA1 channels x {F} L1 frames (cs16), value: samples resident in HBM "
                       "(rewind -> process); k_am: one warp per stream (first, unoptimised AM path)"}
    print(json.dumps(out), flush=True)
    e.close()


def dropin_leg(args):
    """BASELINE configs 1 and 2: ONE stream through the drop-in libnrsc5.so's public API, fed exactly as the reference
    CLI feeds a file (src/main.c:1097-1119: 32 768-byte nrsc5_pipe_samples_cu8 calls, then stop / close), by the C
    driver nrsc5_b200/dropin/bench_pipe.c; the same binary then runs the unmodified reference library (one CPU core)
    on the same bytes.  Config 1 = support/sample.xz, config 2 = a synthetic FM MP1 capture of 8 L1 frames.  The HDC
    packet digest of the two runs must agree.  Prints one JSON object."""
    import lzma
    import tempfile
    exe = os.path.join(ROOT, "nrsc5_b200", "dropin", "_build", "bench_pipe")
    dropin = os.path.join(ROOT, "nrsc5_b200", "dropin", "_build", "libnrsc5.so")
    ref = os.path.join(ROOT, "oracle", "_ref", "libnrsc5_ref.so")
    if not (os.path.exists(exe) and os.path.exists(dropin)):
        print(json.dumps({"error": "drop-in not built (needs the reference tree at build time)"}))
        return
    out = {"what": "nrsc5_open_pipe -> nrsc5_pipe_samples_cu8 in 32768-byte pushes -> nrsc5_stop -> nrsc5_close on one stream; "
                   "wall clock of the push loop + stop + close, best of 8 after one warm-up pass, input in memory",
           "driver": "nrsc5_b200/dropin/bench_pipe.c (the reference CLI's push loop around a dlopen'ed library)"}
    with tempfile.TemporaryDirectory() as td:
        cases = {}
        sample = os.path.join(ROOT, "oracle", "_ref", "sample.xz")
        if os.path.exists(sample):
            path = os.path.join(td, "sample.cu8")
            with open(path, "wb") as f:
                f.write(lzma.open(sample).read())
            cases["config1_sample_xz"] = path
        from nrsc5_b200 import synth
        cap = synth.make_fm_mp1(nframes=8, seed=1234, lead_in=1777, tail_blocks=2)
        path = os.path.join(td, "mp1.cu8")
        cap.cu8[: cap.cu8.size & ~3].tofile(path)
        cases["config2_synthetic_mp1_8_frames"] = path
        for name, path in cases.items():
            res = {}
            for which, lib in (("dropin_b200", dropin), ("reference_cpu_1core", ref)):
                if not os.path.exists(lib):
                    continue
                r = subprocess.run([exe, lib, path, "--reps", "8"], capture_output=True, text=True, timeout=600)
                if r.returncode != 0:
                    res[which] = {"error": (r.stderr or r.stdout)[-300:]}
                    continue
                res[which] = json.loads(r.stdout.strip().splitlines()[-1])
            a, b = res.get("dropin_b200", {}), res.get("reference_cpu_1core", {})
            if "hdc_fnv" in a and "hdc_fnv" in b:
                same = all(a[k] == b[k] for k in ("hdc", "hdc_bytes", "hdc_fnv", "sync", "lost_sync", "mer", "ber", "id3", "audio_service"))
                res["events_identical_to_reference"] = same
                assert same, (name, a, b)
                res["speedup_vs_reference_1core"] = a["x_realtime"] and b["x_realtime"] and a["x_realtime"] / b["x_realtime"]
            out[name] = res
    print(json.dumps(out), flush=True)


def chan_leg(args):
    """SURVEY 8 f3: the wideband channeliser (csrc/channelizer.cu, tcgen05.mma.kind::i8).  One cu8 capture at 23.814 MS/s
    resident in HBM -> 100 FM channels (the whole 88-108 MHz raster) at 744 187.5 S/s cs16, device to device.  Gate: a
    slice of the output equals the numpy restatement bit for bit.  Prints one JSON object."""
    import torch
    from nrsc5_b200 import channelizer as ch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import chan_oracle
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    offs = list(range(-99, 100, 2))                             # 100 channels, 200 kHz apart
    nbytes = 1 << 27                                            # 67.1 M complex samples = 2.82 s of signal, larger than L2
    g = torch.Generator(device=dev)
    g.manual_seed(7)
    cap = torch.randint(0, 256, (nbytes,), dtype=torch.uint8, device=dev, generator=g)
    nout = ch.outputs(nbytes)
    stride = 2 * nout
    out = torch.zeros((len(offs), stride), dtype=torch.int16, device=dev)
    stream = torch.cuda.current_stream()
    with ch.Channelizer(offs) as c:
        taps, ph = c.tables()
        run = lambda: c.run_device(cap.data_ptr(), nbytes, out.data_ptr(), stride, stream.cuda_stream)   # noqa: E731
        run()
        torch.cuda.synchronize()
        part = cap[: 64 * 1500].cpu().numpy()
        want = chan_oracle.channelize(part, offs, taps, ph)
        got = out[:, : want.shape[1]].cpu().numpy()
        assert np.array_equal(got, want), "channeliser output differs from the numpy restatement"
        tail = out[:, 2 * (nout - 64): 2 * nout].cpu().numpy()                   # the end of the capture as well
        want_t = chan_oracle.channelize(cap[nbytes - 64 * (64 + 7):].cpu().numpy(), offs, taps, ph, n0=nout - 64)
        assert np.array_equal(tail, want_t), "channeliser output differs from the numpy restatement at the end of the capture"
        for _ in range(3):
            run()
        torch.cuda.synchronize()
        steps = args.steps
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        for _ in range(steps):
            run()
        ev1.record(stream)
        torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1) / steps
    samples = nbytes // 2
    groups = (len(offs) + 31) // 32
    macs = nout * groups * 128 * 512                           # int8 multiply-accumulates issued (rows of B incl. padding channels)
    useful = nout * len(offs) * 4 * 512
    peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
    bf16 = float(peaks.get("bf16_tflops", 1660.8))
    peak_i8 = 2 * bf16                                          # int8 runs at twice the bf16 rate; no int8 GEMM measurement in MEASURED_PEAKS.json
    hbm, hbm_src = measured_peak()
    traffic = nbytes + len(offs) * nout * 4
    dram = None
    try:                                                   # DRAM bytes of one launch from the ncu capture of this very leg
        tj = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json"))).get("k_channelize")
        dram = tj and (tj["dram_read_bytes"] + tj["dram_write_bytes"])
    except Exception:                                      # noqa: BLE001
        pass
    out_j = {"value": samples / (ms * 1e-3) / 1e6, "unit": "Msamples/s (wideband cu8 complex, 23.814 MS/s)", "ms_per_step": ms,
             "x_realtime": samples / (ms * 1e-3) / 23814000.0, "channels": len(offs), "outputs_per_channel": int(nout), "steps": steps,
             "channel_msamples_per_s": len(offs) * nout / (ms * 1e-3) / 1e6,
             "roofline": {"bound": "tensor", "kernel": "k_channelize (tcgen05.mma.kind::i8, M128 N128 K512 per tile)",
                          "achieved": 2 * macs / (ms * 1e-3) / 1e12, "useful": 2 * useful / (ms * 1e-3) / 1e12, "peak": peak_i8, "unit": "TOP/s",
                          "frac": 2 * macs / (ms * 1e-3) / 1e12 / peak_i8,
                          "peak_source": "2 x MEASURED_PEAKS.json bf16_tflops (int8 tensor rate; no int8 measurement in that file)",
                          "hbm_gbs": traffic / (ms * 1e-3) / 1e9, "hbm_frac": traffic / (ms * 1e-3) / 1e9 / hbm, "algorithmic_bytes": traffic,
                          "traffic": dram, "traffic_source": "profiles/r2_ncu_summary.md (ncu --set full, one launch of this leg)"},
             "parity_gate": {"ok": True, "what": "first 1493 and last 64 output samples of all 100 channels == oracle/chan_oracle.py"},
             "workload": "one 2^27-byte cu8 capture (uniform random bytes) resident in HBM -> 100 channels x %d cs16 samples, device to device" % nout}
    print(json.dumps(out_j), flush=True)


def stream_views(caps, nstreams: int, rank: int):
    """Stream s of this rank = capture (g % D) with the first 4*(37*(g // D) % 1080) bytes dropped,
    g = global stream index: distinct alignments, so distinct acquisition paths."""
    D = len(caps)
    n = min(c.size for c in caps) - 4 * 1080 * 4
    n &= ~63
    views = []
    for s in range(nstreams):
        g = rank * nstreams + s
        off = 4 * ((37 * (g // D)) % 1080)
        views.append(caps[g % D][off: off + n])
    return views, n


# ---------------------------------------------------------------------------
# parity gate: every stream of a timed workload against the CPU oracle (checker only - never timed, never shipped)
# ---------------------------------------------------------------------------
def record_digest(recs):
    """Order-preserving digest of a parsed record stream: (kind, lc, nbits, crc32 of the packed bits) for every L1 PDU."""
    import zlib
    out = []
    for t, r in recs:
        if t == 1:                                    # REC_FRAME (P1 / P3 / P4)
            out.append(("F", r["lc"], r["nbits"], zlib.crc32(r["bits"])))
        elif t == 2:                                  # REC_PIDS
            out.append(("P", 0, 80, zlib.crc32(r["bits"])))
        elif t == 3:
            out.append(("S", r["psmi"], 0, 0))
        elif t == 4:
            out.append(("L", 0, 0, 0))
    return out


def oracle_digests(views, am=False, workers=None):
    """The same digests from the CPU oracle for every view (the unmodified reference when oracle/_ref holds it, else
    the restatement), one decode per DISTINCT view, on a thread pool (the C code releases the GIL)."""
    from concurrent.futures import ThreadPoolExecutor
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import port
    # oracle/nrsc5_oracle*.c (one decoder object per call, so the calls can run on threads); it is pinned record for
    # record to the unmodified reference by tests/test_oracle*.py
    dec = port.decode_am if am else port.decode
    keys, distinct = [], {}
    for v in views:
        k = (v.__array_interface__["data"][0], v.size)
        keys.append(k)
        distinct.setdefault(k, v)
    items = list(distinct.items())
    with ThreadPoolExecutor(max_workers=workers or min(64, os.cpu_count() or 1)) as ex:
        res = list(ex.map(lambda kv: record_digest(dec(np.ascontiguousarray(kv[1])).records), items))
    by_key = {k: r for (k, _), r in zip(items, res)}
    return [by_key[k] for k in keys], "port (oracle/nrsc5_oracle*.c, pinned to the unmodified reference)", len(items)


def parity_gate(views, recs_per_stream, am=False, what=""):
    """Asserts that every stream's L1 PDUs (P1 / P3 / P4 / PIDS, in order, with the sync events) are the oracle's."""
    want, kind, ndistinct = oracle_digests(views, am=am)
    npdu = 0
    for s, (recs, w) in enumerate(zip(recs_per_stream, want)):
        got = record_digest(recs)
        if got != w:
            k = next((i for i, (a, b) in enumerate(zip(got, w)) if a != b), min(len(got), len(w)))
            raise AssertionError(f"{what}: stream {s} differs from the {kind} oracle at record {k}: "
                                 f"engine {got[k:k + 2]} ({len(got)} records) vs oracle {w[k:k + 2]} ({len(w)})")
        npdu += sum(1 for g in got if g[0] in "FP")
    return {"ok": True, "streams_checked": len(views), "distinct_views": ndistinct, "pdus_compared": npdu, "oracle": kind}


DUMP_BUDGET_BYTES = 63 * 10**6           # leaves room for the .npy headers under 64 MB


def dump_outputs(out_dir, recs_per_stream):
    """Writes what a caller of the timed path receives - every stream's parsed records after the last timed step -
    as float arrays under out_dir, one row per record, streams in order:

      frames.npy       float64 [n, 4]  stream, logical channel, nbits, offset of the PDU's first byte in frame_bytes
      frame_bytes.npy  float32 [m]     the packed PDU bytes of those frames, concatenated
      pids.npy         float32 [n, 12] stream, the 10 PDU bytes, CRC verdict (-1: none)
      events.npy       float64 [n, 4]  stream, record type (engine.REC_SYNC / REC_LOST_SYNC / REC_MER / REC_BER), then
                                       frequency offset (Hz), psmi | 0, 0 | lower, upper MER (dB) | channel BER, 0
      streams.npy      float64 [k]     the streams written

    The sparse event kinds share one array, so that the set of files and their shapes do not depend on whether a
    workload happens to lose sync; an array that would still be empty is an error, not an empty file.

    When all streams take more than 63 MB, a fixed sample of streams (a permutation seeded with 0, taken while it
    fits) is written instead, so that two runs with the same arguments write the same streams."""
    from nrsc5_b200 import engine as eng

    def size(recs):
        return 8 + sum(4 * len(r["bits"]) + 32 if t == eng.REC_FRAME else 48 for t, r in recs)

    order = np.random.default_rng(0).permutation(len(recs_per_stream))
    keep, used = [], 0
    for s in order:
        used += size(recs_per_stream[s])
        if used > DUMP_BUDGET_BYTES:
            break
        keep.append(int(s))
    keep.sort()
    frames, frame_bytes, pids, events = [], [], [], []
    nbytes = 0
    for s in keep:
        for t, r in recs_per_stream[s]:
            if t == eng.REC_FRAME:
                frames.append((s, r["lc"], r["nbits"], nbytes))
                frame_bytes.append(np.frombuffer(r["bits"], dtype=np.uint8))
                nbytes += len(r["bits"])
            elif t == eng.REC_PIDS:
                crc = -1 if r["crc_ok"] is None else r["crc_ok"]
                pids.append([s, *r["bits"], crc])
            elif t == eng.REC_SYNC:
                events.append((s, t, r["freq_offset"], r["psmi"]))
            elif t == eng.REC_LOST_SYNC:
                events.append((s, t, 0.0, 0.0))
            elif t == eng.REC_MER:
                events.append((s, t, r["lower"], r["upper"]))
            elif t == eng.REC_BER:
                events.append((s, t, r["cber"], 0.0))
    os.makedirs(out_dir, exist_ok=True)
    arrays = {
        "frames": np.array(frames, dtype=np.float64).reshape(-1, 4),
        "frame_bytes": (np.concatenate(frame_bytes) if frame_bytes else np.zeros(0, np.uint8)).astype(np.float32),
        "pids": np.array(pids, dtype=np.float32).reshape(-1, 12),
        "events": np.array(events, dtype=np.float64).reshape(-1, 4),
        "streams": np.array(keep, dtype=np.float64),
    }
    empty = [name for name, a in arrays.items() if a.size == 0]
    if empty:
        raise RuntimeError(f"--dump-outputs: the last timed step produced no {', '.join(empty)}")
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


class ClockSampler:
    """Samples SM clocks / throttle reasons with one streaming `nvidia-smi -lms` process (the recipe's
    clocks line in B200_PROFILING.md); only the samples taken between mark_begin() and stop() count."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.t_begin = None
        self._proc = None
        self._th = None

    def start(self):
        try:
            self._proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                           "--format=csv,noheader,nounits", "-lms", "50"],
                                          stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self._proc = None
            return

        def run():
            for line in self._proc.stdout:
                self.rows.append((time.perf_counter(), [x.strip() for x in line.strip().split(",")]))
        self._th = threading.Thread(target=run, daemon=True)
        self._th.start()

    def mark_begin(self):
        self.t_begin = time.perf_counter()

    def stop(self):
        t_end = time.perf_counter()
        if self._proc:
            time.sleep(0.06)
            self._proc.terminate()
            try:
                self._proc.wait(timeout=3)
            except Exception:
                self._proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = [r for (ts, r) in self.rows if self.t_begin is None or (self.t_begin <= ts <= t_end + 0.1)]
        if not rows:
            rows = [r for (_, r) in self.rows[-1:]]
        for r in rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for nme, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def cpu_reference_numbers(bufs, nbytes, reps, am=False):
    """The unmodified reference (oracle/_ref/libnrsc5_ref.so) on this host: one PROCESS per channel, each pinned to its
    own physical core (BASELINE.md §3; oracle/refproc.py), 1 core and all physical cores.  Returns (aggregate
    Msamples/s, cores used, dict of details)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import refproc
    import reftap
    mode = reftap.MODE_AM if am else reftap.MODE_FM
    cpus = refproc.physical_cores()
    n = min(len(cpus), len(bufs))
    refproc.bench_processes(bufs[:1], mode=mode, reps=1, cpus=cpus[:1])          # warm-up (page cache, library load)
    t1, _ = refproc.bench_processes(bufs[:1], mode=mode, reps=reps, cpus=cpus[:1])
    tn, n = refproc.bench_processes(bufs[:n], mode=mode, reps=reps, cpus=cpus[:n])
    per = reps * (nbytes // 2)
    info = {"single_core_value": per / t1 / 1e6, "all_cores_value": n * per / tn / 1e6, "processes": n,
            "physical_cores_available": len(cpus), "logical_cpus": os.cpu_count(), "cpu_model": refproc.cpu_model(),
            "fft": refproc.fft_backend(), "viterbi": "SSE (conv_sse.h)", "scaling_efficiency": (n * per / tn) / (n * per / t1),
            "how": "one process per channel pinned to its own physical core (os.sched_setaffinity), input in RAM, "
                   "32768-byte pushes through nrsc5_pipe_samples_cu8 (reference src/main.c:1097-1119)"}
    return n * per / tn / 1e6, n, info


def reference_arm(args, rank: int, world: int):
    """Times the unmodified reference CPU implementation on this host's cores."""
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import reftap
    import port
    cores = os.cpu_count() or 1
    caps = make_captures(args.distinct, args.frames)
    views, n = stream_views(caps, max(1, cores), 0)
    bufs = [np.ascontiguousarray(v) for v in views]
    info = {}
    if reftap.available():
        kind = "reference"
        vals = []
        for _ in range(max(1, args.warmup - 2)):
            cpu_reference_numbers(bufs[:2], n, 1)
        t0 = time.perf_counter()
        for _ in range(args.steps):                     # a step = every physical core decodes one channel once
            v, nproc, info = cpu_reference_numbers(bufs, n, 1)
            vals.append(v)
        total = time.perf_counter() - t0
        val = float(np.median(vals))
    else:
        kind = "port"
        nproc = 1
        t0 = time.perf_counter()
        for _ in range(args.steps):
            port.decode(bufs[0])
        total = time.perf_counter() - t0
        val = args.steps * (n // 2) / total / 1e6
    sample_desc = (f"{nproc} processes (one per physical core, pinned) x 1 channel x {args.frames} frames+2 blocks "
                   f"({n // 2} cu8 samples each) per step; FFT = oracle/shim/fftshim.c (FFTW 3.3.10 not installed); SSE Viterbi")
    line = {
        "impl": "reference", "metric": "cu8 I/Q Msamples/s", "value": val, "unit": "Msamples/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "int16/f32", "data": "synthetic",
        "config": workload_config(args, n),
        "x_realtime": val * 1e6 / SAMPLE_RATE,
        "cpu_baseline": dict({"value": val, "unit": "Msamples/s", "cores": nproc, "kind": kind, "sample": sample_desc}, **info),
        "e2e": {"value": val, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "host_cores": cores,
    }
    print(json.dumps(line), flush=True)


def workload_config(args, nbytes):
    return {"workload": f"{args.streams} independent synthetic FM MP1 hybrid cu8 channels per GPU "
                        f"(BASELINE config 5 shard), {args.frames} L1 frames + 2 blocks each, full chain to L1 PDUs",
            "streams_per_gpu": args.streams, "frames_per_stream": args.frames, "bytes_per_stream": int(nbytes),
            "distinct_captures": args.distinct,
            "l2": "per-GPU input (streams x bytes_per_stream) exceeds the 126 MB L2; no explicit flush"}


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        reference_arm(args, rank, world)
        return
    if args.l2_leg:
        l2_leg(args)
        return
    if args.am_leg:
        am_leg(args)
        return
    if args.mp3_leg:
        mp3_leg(args)
        return
    if args.dropin_leg:
        dropin_leg(args)
        return
    if args.chan_leg:
        chan_leg(args)
        return

    import torch
    import torch.distributed as dist
    import nrsc5_b200
    from nrsc5_b200 import engine as eng

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the engine has no CPU path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    use_dist = world > 1
    if use_dist:
        dist.init_process_group("nccl", device_id=dev)

    S = args.streams
    if args.dbg:
        eng.load_library().nrsc5b_debug_set(args.dbg & 0xff)
    caps = make_captures(args.distinct, args.frames)
    views, nbytes = stream_views(caps, S, rank)
    samples_per_step = S * (nbytes // 2)

    # host side: one pinned slab [S][nbytes]; device side: the same slab resident in HBM
    host = torch.empty((S, nbytes), dtype=torch.uint8).pin_memory()
    hnp = host.numpy()
    for s, v in enumerate(views):
        hnp[s, :] = v
    devbuf = torch.empty((S, nbytes + 64), dtype=torch.uint8, device=dev)
    devbuf[:, :nbytes].copy_(host)
    devbuf[:, nbytes:] = 127
    torch.cuda.synchronize()

    stream = torch.cuda.current_stream()
    log_cap = (args.frames + 1) * (18272 + 64) + 96 * 1024
    e = nrsc5_b200.Engine(nstreams=S, input_capacity=nbytes + 4096, device=local_rank, log_capacity=log_cap)
    e.set_cuda_stream(stream.cuda_stream)
    log_stride = (log_cap + 15) & ~15
    logbuf = torch.zeros((S, log_stride), dtype=torch.uint8, device=dev)   # caller-owned record log, NCCL-gatherable
    e.attach_device_log(logbuf.data_ptr(), log_stride)

    def barrier():
        if use_dist:
            dist.barrier()
        torch.cuda.synchronize()

    def step_resident():
        e.attach_device_input(devbuf.data_ptr(), nbytes + 64, nbytes)
        e.rewind()
        e.process()

    E2E_CHUNKS = 8                                # input arrives in 8 pushes per channel; copy k+1 overlaps compute k
    host_log = torch.empty((S, log_stride), dtype=torch.uint8).pin_memory()
    host_log_np = host_log.numpy()
    cuts = [((nbytes * k // E2E_CHUNKS) & ~3) for k in range(E2E_CHUNKS + 1)]

    def step_e2e():
        e.reset()

        def push(k):                              # one strided copy: chunk k of every channel
            e.push_cu8_all(host.data_ptr() + cuts[k], nbytes, cuts[k + 1] - cuts[k])
        push(0)
        tok = e.push_fence()
        for k in range(E2E_CHUNKS):
            if k + 1 < E2E_CHUNKS:
                push(k + 1)                       # asynchronous, on the engine's copy stream
                nxt = e.push_fence()
                e.process_fence(tok)              # chunk k as soon as it has landed, while chunk k+1 is in flight
                tok = nxt
            else:
                e.process()
        frames = e.drain_all_raw(host_log_np)         # every stream's records: one state copy + one copy per stream
        d2h = sum(int(f.size) for f in frames)
        if use_dist:
            # gather of the decoded L1 PDU / event slabs to rank 0 over NCCL (the only collective on the path)
            lst = [torch.empty_like(logbuf) for _ in range(world)] if rank == 0 else None
            dist.gather(logbuf, lst, dst=0)
        return d2h, frames

    def timed(fn, steps, warmup):
        sampler = ClockSampler(local_rank)
        sampler.start()
        for _ in range(warmup):
            fn()
        barrier()
        sampler.mark_begin()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = e.stats().kernel_launches
        ev0.record(stream)
        out = None
        for _ in range(steps):
            out = fn()
        ev1.record(stream)
        barrier()
        ms = ev0.elapsed_time(ev1)
        l1 = e.stats().kernel_launches
        clocks = sampler.stop()
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        if use_dist:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), l1 - l0, clocks, out

    # ---- correctness gate: EVERY stream's L1 PDUs (P1 + PIDS, in order, with the sync events) must be the CPU
    # ---- oracle's decode of the same view (rank 0: all streams; other ranks: their first 8, to bound host time)
    step_resident()
    recs_all = e.drain_all()
    ncheck = S if rank == 0 else min(S, 8)
    gate = parity_gate(views[:ncheck], recs_all[:ncheck], what="resident step")
    resident_digests = [record_digest(r) for r in recs_all]
    assert all(any(g[0] == "F" for g in d) for d in resident_digests), "a stream decoded no P1 frame"

    # ---- value: device-resident ----
    ms, launches, clocks, _ = timed(step_resident, args.steps, max(args.warmup, 3))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, e.drain_all())
    total_samples = samples_per_step * world * args.steps
    value = total_samples / (ms * 1e-3) / 1e6

    # ---- per-kernel times (separate pass, CUDA events around each launch) ----
    e.set_profiling(True)
    step_resident()
    torch.cuda.synchronize()
    kt = e.kernel_times()
    e.set_profiling(False)
    # where the front-end kernel's SM time goes: average microseconds per stream-block and phase
    clk_mhz = 1965.0
    phases = {k: {"us_per_call": (c / n / clk_mhz) if n else 0.0, "calls": n} for k, (c, n) in e.phase_cycles().items()}
    st = e.stats()
    peak, peak_src = measured_peak()
    blocks_per_step = None
    # blocks processed in the profiled step = demod launches that had work; use stats delta instead
    e.rewind(); e.attach_device_input(devbuf.data_ptr(), nbytes + 64, nbytes)
    b0 = e.stats().blocks
    e.process(); torch.cuda.synchronize()
    b1 = e.stats().blocks
    blocks_per_step = int(b1 - b0) if b1 > b0 else int(b1)
    frames_per_step = int(e.stats().p1_frames)
    p1_fallbacks = int(e.stats().p1_fallbacks)
    kinfo = {}
    # algorithmic bytes (SURVEY §8d): fused front end 299 520 B per stream-block (276 480 B cu8 in + 23 040 B
    # int8 soft bits out); P1 decode group 387 072 B per L1 frame
    alg = {"front": FUSED_BYTES_PER_BLOCK * blocks_per_step, "p1": P1_BYTES_PER_FRAME * frames_per_step}
    for k, v in kt.items():
        gbs = alg[k] / (v["ms"] * 1e-3) / 1e9 if v["ms"] > 0 else 0.0
        kinfo[k] = {"ms_per_step": v["ms"], "launches": v["launches"], "alg_bytes_per_step": alg[k], "achieved_gbs": gbs}
    dom = max(("front", "p1"), key=lambda k: kt[k]["ms"])
    # DRAM traffic of the dominant kernel from the committed ncu --set full capture, scaled to this run's
    # average launch (bytes per stream-block x stream-blocks per launch)
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "r2_traffic.json")
    if not os.path.exists(tp):
        tp = os.path.join(ROOT, "profiles", "r1_traffic.json")
    if dom == "front" and os.path.exists(tp):
        tj = json.load(open(tp))
        per_block = (tj["k_stream"]["dram_read_bytes"] + tj["k_stream"]["dram_write_bytes"]) / tj["k_stream"]["stream_blocks"]
        traffic = per_block * blocks_per_step / max(1, kt[dom]["launches"])
        traffic_src = tj["source"]
    roofline = {"bound": "hbm", "kernel": "k_stream (stream-resident front end: prep+halfband+NCO+FFT+sync+demap)" if dom == "front" else "P1 decode group",
                "achieved": kinfo[dom]["achieved_gbs"], "peak": peak, "unit": "GB/s",
                "frac": kinfo[dom]["achieved_gbs"] / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "alg_bytes_per_launch": alg[dom] / max(1, kt[dom]["launches"]),
                "chain_frac_of_hbm": (2.34 * value * 1e6 / world) / (peak * 1e9),
                "kernels": kinfo, "front_phases_at_1965MHz": phases,
                "p1_frames_per_step": frames_per_step, "p1_fast_path_fallbacks": p1_fallbacks}

    # ---- e2e ----
    e2e = None
    if not args.no_e2e:
        ms2, _, _, out = timed(step_e2e, args.steps, max(args.warmup, 3))
        d2h = out[0] if out else 0
        # the records of the last timed e2e step (host buffers, chunked pushes) must be the resident step's, stream by stream
        e2e_digests = [record_digest(eng.parse_records(f.tobytes())) for f in out[1]]
        assert e2e_digests == resident_digests, "e2e records differ from the device-resident step's"
        gate["e2e_equals_resident"] = True
        e2e_val = total_samples / (ms2 * 1e-3) / 1e6
        # the PCIe floor of this box: the same bytes as one pinned host->device copy, nothing else
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        ev0.record(stream)
        for _ in range(3):
            devbuf[:, :nbytes].copy_(host, non_blocking=True)
        ev1.record(stream)
        torch.cuda.synchronize()
        h2d_ms = ev0.elapsed_time(ev1) / 3
        e2e = {"value": e2e_val, "unit": "Msamples/s", "h2d_bytes_per_step": int(S * nbytes), "d2h_bytes_per_step": int(d2h),
               "ms_per_step": ms2 / args.steps, "x_realtime": e2e_val * 1e6 / SAMPLE_RATE,
               "h2d_copy_alone_ms": h2d_ms, "h2d_copy_alone_gbs": S * nbytes / (h2d_ms * 1e-3) / 1e9}

    # ---- CPU baseline beside it (rank 0, N=1 only): the unmodified reference, one process per channel and core ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import reftap
        bufs = [np.ascontiguousarray(hnp[s]) for s in range(min(S, os.cpu_count() or 1))]
        if reftap.available():
            reps = 2
            v, nproc, info = cpu_reference_numbers(bufs, nbytes, reps)
            cpu = dict({"value": v, "unit": "Msamples/s", "cores": nproc, "kind": "reference",
                        "sample": f"{nproc} processes x {reps} passes over one {nbytes // 2}-sample channel of the bench workload each "
                                  "(unmodified reference, SSE Viterbi, fftshim FFT in place of FFTW)"}, **info)
        else:
            import port
            t0 = time.perf_counter()
            port.decode(bufs[0])
            dt = time.perf_counter() - t0
            cpu = {"value": (nbytes // 2) / dt / 1e6, "unit": "Msamples/s", "cores": 1, "kind": "port",
                   "sample": "one channel, one pass, oracle/nrsc5_oracle.c"}

    # ---- L2 framing on the device (SURVEY 8 f1): separate leg, separate process (rank 0, N=1 only) ----
    l2 = None
    if rank == 0 and world == 1 and not args.no_l2:
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--l2-leg", "--streams", str(S), "--frames", str(args.frames),
                                "--steps", str(args.steps)], capture_output=True, text=True, timeout=600)
            last = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
            l2 = json.loads(last[-1]) if r.returncode == 0 and last else {"error": (r.stderr or r.stdout)[-400:]}
        except Exception as ex:                                    # noqa: BLE001 - the leg must not take the headline down
            l2 = {"error": repr(ex)[:400]}

    # ---- AM, BASELINE config 4 (separate process, rank 0, N=1 only) ----
    am = None
    if rank == 0 and world == 1 and not args.no_am:
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--am-leg", "--am-streams", str(args.am_streams),
                                "--am-frames", str(args.am_frames), "--steps", str(args.steps)],
                               capture_output=True, text=True, timeout=420)
            last = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
            am = json.loads(last[-1]) if r.returncode == 0 and last else {"error": (r.stderr or r.stdout)[-400:]}
        except Exception as ex:                                    # noqa: BLE001
            am = {"error": repr(ex)[:400]}

    # ---- FM MP3, BASELINE config 3 (separate process, rank 0, N=1 only) ----
    mp3 = None
    if rank == 0 and world == 1 and not args.no_mp3:
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--mp3-leg", "--mp3-streams", str(args.mp3_streams),
                                "--mp3-frames", str(args.mp3_frames), "--steps", str(args.steps)],
                               capture_output=True, text=True, timeout=420)
            last = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
            mp3 = json.loads(last[-1]) if r.returncode == 0 and last else {"error": (r.stderr or r.stdout)[-400:]}
        except Exception as ex:                                    # noqa: BLE001
            mp3 = {"error": repr(ex)[:400]}

    # ---- one stream through the drop-in's public API, BASELINE configs 1 and 2 (separate process, rank 0, N=1 only) ----
    dropin = None
    if rank == 0 and world == 1 and not args.no_dropin:
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--dropin-leg"], capture_output=True, text=True, timeout=600)
            last = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
            dropin = json.loads(last[-1]) if r.returncode == 0 and last else {"error": (r.stderr or r.stdout)[-400:]}
        except Exception as ex:                                    # noqa: BLE001
            dropin = {"error": repr(ex)[:400]}

    # ---- the wideband channeliser, SURVEY 8 f3 (separate process, rank 0, N=1 only) ----
    chan = None
    if rank == 0 and world == 1 and not args.no_chan:
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--chan-leg", "--steps", str(args.steps)],
                               capture_output=True, text=True, timeout=420)
            last = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
            chan = json.loads(last[-1]) if r.returncode == 0 and last else {"error": (r.stderr or r.stdout)[-400:]}
        except Exception as ex:                                    # noqa: BLE001
            chan = {"error": repr(ex)[:400]}

    if rank == 0:
        line = {
            "metric": "cu8 I/Q Msamples/s", "value": value, "unit": "Msamples/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8/int16/f32", "data": "synthetic", "config": workload_config(args, nbytes),
            "x_realtime": value * 1e6 / SAMPLE_RATE, "x_realtime_per_gpu": value * 1e6 / SAMPLE_RATE / world,
            "clocks": clocks, "gpu_launches": int(launches), "roofline": roofline, "parity_gate": gate,
        }
        if e2e:
            line["e2e"] = e2e
        if cpu:
            line["cpu_baseline"] = cpu
        if l2:
            line["l2_on_device"] = l2
        if am:
            line["am_config4"] = am
        if mp3:
            line["mp3_config3"] = mp3
        if dropin:
            line["single_stream_dropin"] = dropin
        if chan:
            line["channeliser_f3"] = chan
        print(json.dumps(line), flush=True)
    e.close()
    if use_dist:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
