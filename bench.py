#!/usr/bin/env python3
"""bench.py -- throughput of the batched Opus decode hot path on B200.

Workload (BASELINE.json configs[1]): 4096 CELT-only fullband 20 ms stereo streams @64 kbps
(160-byte packets, TOC 0xFC) per GPU; one "step" decodes one packet of every stream in two launches:
k_synth_rangedec (one lane per packet: every range-coded symbol) and k_frame_w (one warp per stream:
PVQ expansion -> IMDCT + TDAC overlap-add -> comb post-filter -> interleaved PCM store, nothing in
between leaves the SM).  Streams are independent, so N GPUs each own their own 4096 streams (weak
scaling, no collective on the data path).

  value  : concurrent realtime streams = stereo frames decoded per second x 0.020 s, whole job,
           packets already resident in HBM, PCM left in the device ring (CUDA events, max over ranks)
  e2e    : the same metric through the host-buffer entry point (BatchDecoder.decode_float):
           pinned host packets -> H2D -> decode -> D2H float PCM inside the timed region
  roofline: the frame kernel, algorithmic bytes 4*(2*960+120) per channel-frame (SURVEY.md 8d) plus the
           4*(T+2) bytes of comb history of every channel-frame the post-filter ran on / average launch time
  cpu_baseline / --impl reference: the CPU oracle (a C port of the reference crate's code for this
           path; the crate itself is Rust and cannot be built in this image) on the host cores.

One JSON line on stdout (rank 0).
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LM, CHANNELS, PKT_BYTES, NF = 3, 2, 160, 960
FRAME_S = 0.020
ALGO_BYTES_PER_CHANNEL_FRAME = 4 * (2 * NF + 120)  # SURVEY.md 8d: coeffs + carry in, PCM + carry out


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock and throttle reasons polled through NVML every few milliseconds, only while a timed
    region is open (`with sampler.region():`), so the median is a median under load."""
    REASONS = (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40))

    def __init__(self, index):
        self.index, self.sm, self.mask, self.max_mhz = index, [], 0, None
        self.open, self.quit, self.thread, self.h, self.nv = False, False, None, None, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
        except Exception:
            self.nv = None

    def _poll(self):
        nv = self.nv
        while not self.quit:
            if self.open:
                try:
                    self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                    self.mask |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                except Exception:
                    pass
            time.sleep(0.002)

    class _Region:
        def __init__(self, s):
            self.s = s

        def __enter__(self):
            self.s.open = True

        def __exit__(self, *a):
            self.s.open = False

    def region(self):
        return ClockSampler._Region(self)

    def stop(self):
        self.quit = True
        if self.thread:
            self.thread.join(timeout=1.0)
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(n for n, bit in self.REASONS if self.mask & bit), "samples": len(self.sm),
                "how": "NVML polled every ~2 ms inside the timed regions (resident, per-kernel and end-to-end passes)"}


def workload_config(n, transient_permille, bitstream=1):
    """The `config` object of both arms (identical by construction)."""
    return {"workload": f"{n} CELT-only fullband 20 ms stereo streams @64 kbps per GPU (BASELINE configs[1]; SYNTH-CELT/{bitstream}, "
                        "160 B packets): range decode + PVQ + IMDCT/TDAC + comb post-filter",
            "streams_per_gpu": n, "frames_per_step_per_gpu": n, "packet_bytes": PKT_BYTES, "frame_ms": 20, "channels": CHANNELS,
            "transient_permille": transient_permille}


def pin_rank_to_cpus(local, world):
    """All GPUs of these boxes hang off one CPU set; give every rank its own slice of it, so that the ranks' feeder
    threads (packet synthesis, the copy-issuing thread, the checksum) do not migrate onto each other."""
    try:
        cpus = sorted(os.sched_getaffinity(0))
        per = max(1, len(cpus) // max(1, world))
        mine = cpus[local * per:(local + 1) * per] or cpus
        os.sched_setaffinity(0, mine)
        return mine
    except Exception:
        return None


def cpu_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def run_reference(args):
    """--impl reference: the CPU implementation of the same path, all host threads, same config/metric.
    Nothing of the product is loaded here: the packets come from the oracle's own range encoder."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = args.streams
    cores = cpu_threads()
    total = args.steps + args.warmup
    packets = O.synth_fill(0, n, 0, total, LM, CHANNELS, PKT_BYTES, args.transient_permille, n_threads=cores)
    L = O.lib()
    x = ctypes.c_uint32(0)
    # Frames are chained per stream (overlap carry, comb history), exactly like the GPU steps: the
    # timed call walks every stream through `steps` consecutive packets; ms_per_step = time / steps.
    if args.warmup:
        L.orc_synth_bench(O.ptr(packets[:args.warmup]), n, args.warmup, PKT_BYTES, LM, CHANNELS, 1, cores, None, ctypes.byref(x))
    t = L.orc_synth_bench(O.ptr(packets[args.warmup:]), n, args.steps, PKT_BYTES, LM, CHANNELS, 1, cores, None, ctypes.byref(x))
    fps = n * args.steps / t
    value = fps * FRAME_S
    line = {
        "impl": "reference", "metric": "concurrent_realtime_48k_streams_decoded", "value": value, "unit": "streams",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32+f32", "data": "synthetic",
        "config": workload_config(n, args.transient_permille, args.bitstream),
        "cpu_baseline": {"value": value, "unit": "streams", "cores": cores, "kind": "port",
                         "sample": f"{args.steps} chained steps x {n} stereo 20 ms frames (the full workload step), "
                                   "C oracle port of the reference crate (Rust toolchain absent), one thread per core"},
        "e2e": {"value": value, "unit": "streams", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


MIX_WEIGHTS = (0.10, 0.10, 0.30, 0.50)      # 2.5 / 5 / 10 / 20 ms
MIX_PKT_BYTES = (64, 80, 112, 160)          # the SYNTH-CELT/1 schedule's sizes per frame length (its bit demand is fixed per LM)


def run_mix(args):
    """--mix: BASELINE configs[4] shape, CELT part, device-resident.  Every step every stream holds a single-frame packet of
    a frame size drawn anew (10/10/30/50 % of 2.5/5/10/20 ms), 10 % of the frames transient; the step's buckets are built on the
    device (OPN_FLAG_MIXED_FRAMES).  The metric is the same: audio seconds decoded per wall-clock second = concurrent
    realtime streams.  An extra line kept under profiles/, not the headline."""
    import torch
    import opus_native_b200 as opn
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libopusb200 has no CPU fallback")
    pin_rank_to_cpus(local, world)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    n, K, W = args.streams, args.steps, args.warmup
    total = K + W
    tp = args.transient_permille if args.transient_permille else 100
    lo, _ = opn.shard_range(n * world, rank, world)
    rnd = np.random.default_rng(1234 + rank)
    stride = max(MIX_PKT_BYTES)
    arena = np.zeros((total, n, stride), np.uint8)
    lens = np.zeros((total, n), np.int32)
    lm_of = rnd.choice(4, size=(total, n), p=MIX_WEIGHTS)
    cores = cpu_threads()
    for f in range(total):
        for lm in range(4):
            ids = np.nonzero(lm_of[f] == lm)[0]
            if len(ids):
                arena[f, ids, :MIX_PKT_BYTES[lm]] = opn.synth_fill(lo + 7 * lm, len(ids), f, 1, lm, CHANNELS, MIX_PKT_BYTES[lm], tp, n_threads=cores)[0]
                lens[f, ids] = MIX_PKT_BYTES[lm]
    audio_s = float((120 << lm_of[W:]).sum()) / 48000.0  # decoded in the timed steps, this rank
    dec = opn.BatchDecoder(n, opn.DecoderConfiguration(48000, CHANNELS, 0), device=local, bitstream=1)
    stream = torch.cuda.ExternalStream(dec.cuda_stream, device=dev)
    d_arena = torch.from_numpy(arena.reshape(-1)).to(dev)
    d_off = (torch.arange(n, dtype=torch.int64, device=dev) * stride).to(torch.int32)
    d_len = torch.from_numpy(lens).to(dev)
    d_res = torch.zeros(n, dtype=torch.int32, device=dev)
    flags = opn.FLAG_DEVICE_PTRS | opn.FLAG_NO_PCM_COPY | opn.FLAG_INPUTS_READY | opn.FLAG_MIXED_FRAMES
    p_arena, p_off, p_len, p_res = d_arena.data_ptr(), d_off.data_ptr(), d_len.data_ptr(), d_res.data_ptr()

    host_s = [0.0]

    def step(f):
        dec.decode_float_ptrs(p_arena + f * n * stride, p_off, p_len + 4 * f * n, None, 0, NF, p_res, flags)

    def timed(k0, k1):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record()
            h0 = time.perf_counter()
            for f in range(k0, k1):
                step(f)
            host_s[0] = time.perf_counter() - h0
            dec.join()
            e1.record()
        dec.synchronize()
        barrier()
        return e0.elapsed_time(e1) * 1e-3

    for f in range(W):
        step(f)
    dec.synchronize()
    assert bool((d_res.cpu().numpy() == (120 << lm_of[W - 1])).all()), "decode reported errors"
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    dec.stats(reset=True)
    with sampler.region():
        t = timed(W, total)
    if dist is not None:
        tt = torch.tensor([t], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t = float(tt.item())
        aa = torch.tensor([audio_s], dtype=torch.float64, device=dev)
        dist.all_reduce(aa, op=dist.ReduceOp.SUM)
        audio_s = float(aa.item())
    launches = sum(dec.stats(reset=True)["launches"])
    host_enqueue_ms = 1e3 * host_s[0] / K
    assert bool((d_res.cpu().numpy() == (120 << lm_of[total - 1])).all())
    dec.reset()
    dec.enable_timing(True)
    for f in range(W):
        step(f)
    dec.stats(reset=True)
    timed(W, total)
    st = dec.stats(reset=True)
    dec.enable_timing(False)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0:
        emit({
            "metric": "concurrent_realtime_48k_streams_decoded", "value": audio_s / t, "unit": "streams", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": 1e3 * t / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32+f32", "data": "synthetic",
            "config": {"workload": f"{n} CELT-only stereo streams per GPU, every packet's frame size drawn 10/10/30/50 % from 2.5/5/10/20 ms "
                                   f"({MIX_PKT_BYTES} B packets, SYNTH-CELT/1), {tp / 10:.0f} % transient frames (BASELINE configs[4] shape, CELT part); "
                                   "device-resident, buckets built on the device (OPN_FLAG_MIXED_FRAMES)",
                       "streams_per_gpu": n, "frames_per_step_per_gpu": n, "channels": CHANNELS, "transient_permille": tp,
                       "mean_frame_ms": 1e3 * audio_s / (world * n * K)},
            "detail": {"per_kernel_ms": {"k_synth_rangedec": st["ms"][0] / K, "k_frame_mix (one launch per group)": st["ms"][1] / K},
                       "frames_per_s": world * n * K / t,
                       "host_enqueue_ms_per_step": host_enqueue_ms},
            "gpu_launches": int(launches), "clocks": clocks,
        })
    if dist is not None:
        dist.destroy_process_group()


SILK_PKT_BYTES = 80   # SILK wideband mono 20 ms at 32 kbps (TOC + SYNTH-SILK/1 payload)


def run_silk(args):
    """--silk: BASELINE configs[2], "16384 SILK-only wideband 16 kHz 20 ms streams: LPC synthesis + resample to 48 kHz on 1
    B200" (SYNTH-SILK/1, DESIGN.md section 3c; mono, 80-byte packets).  Device-resident steps for `value`, the host-buffer
    call for `e2e`, the oracle's CPU loop on a bounded sample for `cpu_baseline`.  An extra line kept under profiles/."""
    import torch
    import opus_native_b200 as opn
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libopusb200 has no CPU fallback")
    pin_rank_to_cpus(local, world)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    n, K, W = args.streams, args.steps, args.warmup
    total = K + W
    nb, n48, ch = SILK_PKT_BYTES, 960, 1
    lo, _ = opn.shard_range(n * world, rank, world)
    cores = cpu_threads()
    packets = opn.silk_fill(lo, n, 0, total, 2, 20, ch, nb, n_threads=cores)
    bits = opn.BITSTREAM_SYNTH_CELT_1 | opn.BITSTREAM_SYNTH_SILK_1
    dec = opn.BatchDecoder(n, opn.DecoderConfiguration(48000, ch, 0), device=local, bitstream=bits)
    stream = torch.cuda.ExternalStream(dec.cuda_stream, device=dev)
    d_arena = torch.from_numpy(packets.reshape(-1)).to(dev)
    d_off = (torch.arange(n, dtype=torch.int64, device=dev) * nb).to(torch.int32)
    d_len = torch.full((n,), nb, dtype=torch.int32, device=dev)
    d_res = torch.zeros(n, dtype=torch.int32, device=dev)
    flags = opn.FLAG_DEVICE_PTRS | opn.FLAG_NO_PCM_COPY | opn.FLAG_INPUTS_READY | opn.FLAG_SILK_FRAMES
    p_arena, p_off, p_len, p_res = d_arena.data_ptr(), d_off.data_ptr(), d_len.data_ptr(), d_res.data_ptr()
    host_s = [0.0]

    def step(f):
        dec.decode_float_ptrs(p_arena + f * n * nb, p_off, p_len, None, 0, n48, p_res, flags)

    def timed(k0, k1):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record()
            h0 = time.perf_counter()
            for f in range(k0, k1):
                step(f)
            host_s[0] = time.perf_counter() - h0
            dec.join()
            e1.record()
        dec.synchronize()
        barrier()
        return e0.elapsed_time(e1) * 1e-3

    for f in range(W):
        step(f)
    dec.synchronize()
    assert int((d_res != n48).sum().item()) == 0, "decode reported errors"
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    dec.stats(reset=True)
    with sampler.region():
        t = max_over_ranks(timed(W, total))
    launches = sum(dec.stats(reset=True)["launches"])
    host_enqueue_ms = 1e3 * host_s[0] / K
    dec.reset()
    dec.enable_timing(True)
    for f in range(W):
        step(f)
    dec.stats(reset=True)
    with sampler.region():
        timed(W, total)
    st = dec.stats(reset=True)
    dec.enable_timing(False)
    k0_ms, k1_ms = st["ms"][0] / K, st["ms"][1] / K

    # end to end: pinned host packets in, pinned host PCM out, two calls in flight
    dec2 = opn.BatchDecoder(n, opn.DecoderConfiguration(48000, ch, 0), device=local, bitstream=bits)
    h_arena = torch.from_numpy(packets.reshape(-1)).pin_memory()
    h_pcm = [torch.zeros((n, n48 * ch), dtype=torch.float32).pin_memory() for _ in range(2)]
    a_np, p_np = h_arena.numpy(), [x.numpy() for x in h_pcm]
    offs = (np.arange(n, dtype=np.uint32) * nb)
    lens = np.full(n, nb, np.uint32)
    res = [np.zeros(n, np.int32) for _ in range(2)]

    def run_e2e(k0, k1):
        probe, ticket = 0.0, None
        for f in range(k0, k1):
            q = f & 1
            tk = dec2.decode_float_ptrs(a_np.ctypes.data + f * n * nb, offs.ctypes.data, lens.ctypes.data, p_np[q].ctypes.data, n48 * ch, n48,
                                        res[q].ctypes.data, opn.FLAG_SUBMIT_ONLY)
            if ticket is not None:
                dec2.wait(ticket)
                probe += float(p_np[(f - 1) & 1][0, 0]) + float(p_np[(f - 1) & 1][-1, -1])
            ticket = tk
        dec2.wait(ticket)
        return probe + float(p_np[(k1 - 1) & 1][0, 0]) + float(p_np[(k1 - 1) & 1][-1, -1])

    Ke = min(K, 50)
    run_e2e(0, W)
    barrier()
    with sampler.region():
        h0 = time.perf_counter()
        checksum = run_e2e(W, W + Ke)
        t_e2e = max_over_ranks(time.perf_counter() - h0)
    assert all(int((r != n48).sum()) == 0 for r in res)
    clocks = sampler.stop() if rank == 0 else None

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_lib as O
        ns, nfr = min(n, 2048), min(total, 25)
        x = ctypes.c_uint32(0)
        sample = np.ascontiguousarray(packets[:nfr, :ns])
        tc = O.lib().orc_silk_bench(O.ptr(sample), ns, nfr, nb, 2, 20, ch, cores, None, ctypes.byref(x))
        cpu = {"value": ns * nfr / tc * FRAME_S, "unit": "streams", "cores": cores, "kind": "port",
               "sample": f"{nfr} chained frames x {ns} streams of the same packets, C oracle (oracle/silk.c), one thread per core, {tc:.2f} s wall"}
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, dec, n, n48, ch, dev)
    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        chan_frames = n * ch
        # per channel-frame: 3840 B of PCM out, the 144-byte side record in, the filter state in and out (sLPC 64, A_Q12 32,
        # gain 4, resampler 32), the excitation history read by the long-term predictor and written back (1280 each)
        algo = chan_frames * (3840 + 144 + 2 * 132 + 2 * 1280)
        emit({
            "metric": "concurrent_realtime_48k_streams_decoded", "value": world * n * K / t * FRAME_S, "unit": "streams", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": 1e3 * t / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "i32+f32", "data": "synthetic",
            "config": {"workload": f"{n} SILK-only wideband (16 kHz internal) 20 ms mono streams per GPU (BASELINE configs[2]; SYNTH-SILK/1, "
                                   f"{nb} B packets): range decode + PVQ shell blocks + long-term prediction + integer LPC synthesis + "
                                   "polyphase resampler to 48 kHz",
                       "streams_per_gpu": n, "frames_per_step_per_gpu": n, "packet_bytes": nb, "frame_ms": 20, "channels": ch},
            "detail": {"cache": f"{total} distinct packet sets resident in HBM, each read once; every step writes {n * 3840 / 1e6:.1f} MB of PCM",
                       "per_kernel_ms": {"k_silk_rangedec": k0_ms, "k_silk_frame": k1_ms}, "host_enqueue_ms_per_step": host_enqueue_ms,
                       "e2e_checksum": checksum, "peak_source": peak_src},
            "e2e": {"value": world * n * Ke / t_e2e * FRAME_S, "unit": "streams", "h2d_bytes_per_step": n * nb + 4 * 4 * n,
                    "d2h_bytes_per_step": n * n48 * ch * 4, "ms_per_step": 1e3 * t_e2e / Ke, "steps": Ke},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": "k_silk_frame<1,1> (excitation + LTP + LPC synthesis across streams + resampler + PCM store)",
                         "achieved": algo / (k1_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s", "frac": algo / (k1_ms * 1e-3) / 1e9 / peak,
                         "traffic": 15835904.0,
                         "traffic_source": "static: profiles/r2b_silk_frame_ncu_summary.json, 2026-10-19: ncu --set full, dram__bytes_read.sum + "
                                           "dram__bytes_write.sum summed over the three k_silk_frame<1,1> launches of one 16384-stream step; well below "
                                           "the algorithmic bytes because packets' records, filter state and the 62.9 MB of PCM a step writes live in the "
                                           "126 MB L2 between launches (ncu flushes before each launch: what is left is read traffic)",
                         "algorithmic_bytes_per_launch": algo,
                         "bytes_note": "per channel-frame: 3840 B PCM + 144 B side record + 2 x 132 B filter state + 2 x 1280 B excitation history"},
            "cpu_baseline": cpu, "clocks": clocks,
        })
    if dist is not None:
        dist.destroy_process_group()


_REAL_STDOUT = None


def quiet_stdout():
    """The contract is ONE JSON line on stdout: route everything native libraries print there (NCCL's
    version banner, for one) to stderr and keep the real stdout for the result line."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


DUMP_BYTES = 64_000_000  # array data written by --dump-outputs at most


class _DeviceArray:
    """A device pointer the library hands out, in the form torch.as_tensor reads (__cuda_array_interface__)."""

    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"data": (ptr, False), "shape": shape, "typestr": typestr, "version": 2}


def dump_outputs(out_dir, dec, n, frame, channels, dev):
    """--dump-outputs: what a caller of the device-resident path receives after the last timed step, as .npy files:
    pcm [streams, frame * channels] float32 (interleaved; read from the decoder's PCM ring, where the step's frame ends at
    each stream's ring position), final_range [streams] (the range coder's final state per stream, exact in float64) and
    stream [streams] (stream ids).  Above DUMP_BYTES a fixed, seeded sample of the streams is written."""
    import torch
    per_stream = frame * channels * 4 + 8 + 8
    k = min(n, DUMP_BYTES // per_stream)
    ids = np.arange(n) if k == n else np.sort(np.random.default_rng(0).choice(n, k, replace=False))
    ring_ptr, ring_n, pos_ptr = dec.ring()
    ring = torch.as_tensor(_DeviceArray(ring_ptr, (n, ring_n, channels), "<f4"), device=dev)
    pos = torch.as_tensor(_DeviceArray(pos_ptr, (n,), "<i4"), device=dev).long()
    sel = torch.from_numpy(ids).to(dev)
    idx = (pos[sel, None] - frame + torch.arange(frame, device=dev)) % ring_n
    pcm = torch.gather(ring[sel], 1, idx[:, :, None].expand(-1, -1, channels)).reshape(k, frame * channels)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "pcm.npy"), pcm.cpu().numpy())
    np.save(os.path.join(out_dir, "final_range.npy"), dec.final_ranges()[ids].astype(np.float64))
    np.save(os.path.join(out_dir, "stream.npy"), ids.astype(np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--streams", type=int, default=4096, help="streams per GPU (BASELINE config 2: 4096)")
    ap.add_argument("--transient-permille", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--bitstream", type=int, default=1, choices=[1, 2],
                    help="1: SYNTH-CELT/1 (the headline workload), 2: SYNTH-CELT/2 (allocation-driven frames; kept next to it under profiles/)")
    ap.add_argument("--mix", action="store_true",
                    help="extra workload: per-packet frame sizes 2.5-20 ms with transients, device-resident (BASELINE configs[4] shape, CELT part)")
    ap.add_argument("--silk", action="store_true",
                    help="extra workload: BASELINE configs[2], SILK-only wideband 20 ms mono streams (SYNTH-SILK/1), default 16384 streams")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps write the last step's outputs (PCM, final range per stream) as DIR/<name>.npy, "
                         "rank 0; the inputs are the same in every run with the same arguments")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    if args.dump_outputs and (args.mix or args.impl != "b200"):
        raise SystemExit("--dump-outputs covers the b200 arm's fixed-frame workloads (the default and --silk)")
    quiet_stdout()
    if args.silk:
        if args.impl != "b200":
            raise SystemExit("--silk is an extra line of the b200 arm")
        if args.streams == 4096:
            args.streams = 16384
        run_silk(args)
        return
    if args.mix:
        if args.impl != "b200":
            raise SystemExit("--mix is an extra line of the b200 arm")
        run_mix(args)
        return
    if args.impl == "reference":
        if args.bitstream != 1:
            raise SystemExit("--impl reference times the SYNTH-CELT/1 workload (the headline); there is no CPU loop for --bitstream 2")
        run_reference(args)
        return

    import torch
    import opus_native_b200 as opn

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libopusb200 has no CPU fallback")
    cpus = pin_rank_to_cpus(local, world)  # before any allocation: pinned buffers and threads stay on this rank's cores
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    n = args.streams
    K, W = args.steps, args.warmup
    total = K + W
    lo, hi = opn.shard_range(n * world, rank, world)  # this rank's global stream ids
    cores = cpu_threads()  # this rank's share after pinning
    fill = opn.synth_fill if args.bitstream == 1 else opn.celt2_fill
    packets = fill(lo, n, 0, total, LM, CHANNELS, PKT_BYTES, args.transient_permille, n_threads=cores)
    step_bytes = n * PKT_BYTES

    # ---------------- resident-input measurement (value) ----------------
    dec = opn.BatchDecoder(n, opn.DecoderConfiguration(48000, CHANNELS, 0), device=local, bitstream=args.bitstream)
    stream = torch.cuda.ExternalStream(dec.cuda_stream, device=dev)
    d_arena = torch.from_numpy(packets.reshape(-1)).to(dev)
    d_off = (torch.arange(n, dtype=torch.int64, device=dev) * PKT_BYTES).to(torch.int32)
    d_len = torch.full((n,), PKT_BYTES, dtype=torch.int32, device=dev)
    d_res = torch.zeros(n, dtype=torch.int32, device=dev)
    flags = opn.FLAG_DEVICE_PTRS | opn.FLAG_NO_PCM_COPY | opn.FLAG_INPUTS_READY  # packets are resident: the range decode may run up to 8 steps ahead

    p_arena, p_off, p_len, p_res = d_arena.data_ptr(), d_off.data_ptr(), d_len.data_ptr(), d_res.data_ptr()

    host_s = [0.0]

    def step_resident(f):
        dec.decode_float_ptrs(p_arena + f * step_bytes, p_off, p_len, None, 0, NF, p_res, flags)

    def timed_resident(k0, k1):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record()
            h0 = time.perf_counter()
            for f in range(k0, k1):
                step_resident(f)
            host_s[0] = time.perf_counter() - h0  # host time to enqueue the steps (asynchronous calls)
            dec.join()  # two thirds of the streams' frame kernels run on internal streams: make them ancestors of e1
            e1.record()
        dec.synchronize()
        barrier()
        return e0.elapsed_time(e1) * 1e-3

    for f in range(W):
        step_resident(f)
    dec.synchronize()
    assert int((d_res != NF).sum().item()) == 0, "decode reported errors"
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    dec.stats(reset=True)
    with sampler.region():
        t_value = max_over_ranks(timed_resident(W, total))
    launches = sum(dec.stats(reset=True)["launches"])
    host_enqueue_ms = 1e3 * host_s[0] / K
    # same K steps again with cudaEvents around every kernel launch -> per-kernel durations
    dec.reset()
    dec.enable_timing(True)
    for f in range(W):
        step_resident(f)
    dec.stats(reset=True)
    with sampler.region():
        timed_resident(W, total)
    st = dec.stats(reset=True)
    dec.enable_timing(False)
    k0_ms, k1_ms, k2_ms = st["ms"][0] / K, st["ms"][1] / K, st["ms"][2] / K
    hist_samples = dec.history_samples(reset=True) / K  # per launch: sum over channel-frames of max(T0,T1)+2
    assert int((d_res != NF).sum().item()) == 0

    # ---------------- end-to-end through the host-buffer API ----------------
    # The call a user makes: pinned host packets in, pinned host PCM out, every step.  Two calls are kept
    # in flight (OPN_FLAG_SUBMIT_ONLY + opn_batch_wait), so the 31.5 MB PCM download of step n overlaps the
    # upload and decode of step n+1; each step's PCM is read on the host (checksum) after its wait.
    dec2 = opn.BatchDecoder(n, opn.DecoderConfiguration(48000, CHANNELS, 0), device=local, bitstream=args.bitstream)
    h_arena = torch.from_numpy(packets.reshape(-1)).pin_memory()
    h_pcm = [torch.zeros((n, NF * CHANNELS), dtype=torch.float32).pin_memory() for _ in range(2)]
    a_np, p_np = h_arena.numpy(), [t.numpy() for t in h_pcm]
    offs = (np.arange(n, dtype=np.uint32) * PKT_BYTES)
    lens = np.full(n, PKT_BYTES, np.uint32)
    res = [np.zeros(n, np.int32) for _ in range(2)]

    def submit_e2e(f):
        q = f & 1
        return dec2.decode_float_ptrs(a_np.ctypes.data + f * step_bytes, offs.ctypes.data, lens.ctypes.data, p_np[q].ctypes.data,
                                      NF * CHANNELS, NF, res[q].ctypes.data, opn.FLAG_SUBMIT_ONLY)

    def run_e2e(k0, k1):
        probe, ticket = 0.0, None
        for f in range(k0, k1):
            t = submit_e2e(f)
            if ticket is not None:
                dec2.wait(ticket)
                probe += float(p_np[(f - 1) & 1][0, 0]) + float(p_np[(f - 1) & 1][-1, -1])  # the result is read on the host
            ticket = t
        dec2.wait(ticket)
        probe += float(p_np[(k1 - 1) & 1][0, 0]) + float(p_np[(k1 - 1) & 1][-1, -1])
        return probe

    # plain pinned D2H copies of one step's PCM (31.5 MB), all ranks at once: the ceiling the e2e figure is read against
    probe_src = torch.empty(n * NF * CHANNELS, dtype=torch.float32, device=dev)
    probe_dst = h_pcm[0].view(-1)
    for _ in range(3):
        probe_dst.copy_(probe_src, non_blocking=True)
    barrier()
    pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pe0.record()
    for _ in range(20):
        probe_dst.copy_(probe_src, non_blocking=True)
    pe1.record()
    torch.cuda.synchronize()
    t_probe = max_over_ranks(pe0.elapsed_time(pe1) * 1e-3 / 20)
    pcie_gbs = probe_src.numel() * 4 / t_probe / 1e9  # per GPU, slowest rank
    del probe_src

    run_e2e(0, W)
    barrier()
    with sampler.region():
        t0 = time.perf_counter()
        run_e2e(W, total)
        torch.cuda.synchronize()
        t_e2e = max_over_ranks(time.perf_counter() - t0)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    assert np.all(res[0] == NF) and np.all(res[1] == NF)
    checksum = float(np.abs(p_np[(total - 1) & 1]).sum())

    # ---------------- the same end-to-end loop through Decoder::decode::<i16> (extra figure, not the headline) ----
    # soft clip + Sample::from_f32 run on the device, so half the bytes cross PCIe.
    K16 = min(K, 100)
    dec3 = opn.BatchDecoder(n, opn.DecoderConfiguration(48000, CHANNELS, 0), device=local, bitstream=args.bitstream)
    h_pcm16 = [torch.zeros((n, NF * CHANNELS), dtype=torch.int16).pin_memory() for _ in range(2)]
    p16 = [t.numpy() for t in h_pcm16]

    def run_e2e_i16(k0, k1):
        ticket = None
        for f in range(k0, k1):
            q = f & 1
            t = dec3.decode_i16_ptrs(a_np.ctypes.data + f * step_bytes, offs.ctypes.data, lens.ctypes.data, p16[q].ctypes.data,
                                     NF * CHANNELS, NF, res[q].ctypes.data, opn.FLAG_SUBMIT_ONLY)
            if ticket is not None:
                dec3.wait(ticket)
            ticket = t
        dec3.wait(ticket)

    run_e2e_i16(0, W)
    barrier()
    t0 = time.perf_counter()
    run_e2e_i16(W, W + K16)
    torch.cuda.synchronize()
    t_e2e16 = max_over_ranks(time.perf_counter() - t0)
    barrier()
    assert np.all(res[0] == NF) and np.all(res[1] == NF) and int(np.abs(p16[(W + K16 - 1) & 1].astype(np.int32)).sum()) > 0

    # ---------------- the same loop with ordinary pageable caller memory (extra figure) ----------------
    # What a Rust Vec<f32> / &mut [f32] is: the CUDA runtime stages such copies through its own bounce buffer,
    # synchronously, so calls cannot overlap.  opn_host_alloc / opn_host_register give a caller the pinned kind.
    KP = min(K, 30)
    dec4 = opn.BatchDecoder(n, opn.DecoderConfiguration(48000, CHANNELS, 0), device=local, bitstream=args.bitstream)
    pg_arena = packets.reshape(-1)
    pg_pcm = np.zeros((n, NF * CHANNELS), np.float32)
    for f in range(W):
        dec4.decode_float_ptrs(pg_arena.ctypes.data + f * step_bytes, offs.ctypes.data, lens.ctypes.data, pg_pcm.ctypes.data, NF * CHANNELS,
                               NF, res[0].ctypes.data, 0)
    barrier()
    t0 = time.perf_counter()
    for f in range(W, W + KP):
        dec4.decode_float_ptrs(pg_arena.ctypes.data + f * step_bytes, offs.ctypes.data, lens.ctypes.data, pg_pcm.ctypes.data, NF * CHANNELS,
                               NF, res[0].ctypes.data, 0)
    t_pg = max_over_ranks(time.perf_counter() - t0)
    barrier()
    assert np.all(res[0] == NF) and float(np.abs(pg_pcm).sum()) > 0

    # ---------------- CPU baseline (rank 0, N = 1 only) ----------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and args.bitstream == 1:  # the CPU loop restates SYNTH-CELT/1 only
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_lib as O
        fr = min(total, 48)
        x = ctypes.c_uint32(0)
        tc, reps = 0.0, 0
        while tc < 10.0 and reps < 400:  # about 10 s of wall clock on all cores: the same chained block of frames, decoded again and again
            tc += O.lib().orc_synth_bench(O.ptr(packets[:fr]), n, fr, PKT_BYTES, LM, CHANNELS, 1, cores, None, ctypes.byref(x))
            reps += 1
        cpu = {"value": n * fr * reps / tc * FRAME_S, "unit": "streams", "cores": cores, "kind": "port",
               "sample": f"{reps} passes over {fr} chained frames x {n} streams of the same packets, C oracle port of the reference crate "
                         f"(range decode + PVQ + IMDCT + comb filter), one thread per core, {tc:.1f} s wall"}

    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, dec, n, NF, CHANNELS, dev)
    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        ch_frames = n * CHANNELS
        algo_bytes = ch_frames * ALGO_BYTES_PER_CHANNEL_FRAME + 4 * hist_samples
        achieved = algo_bytes / (k1_ms * 1e-3) / 1e9
        value = world * n * K / t_value * FRAME_S
        e2e = world * n * K / t_e2e * FRAME_S
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            try:
                tj = json.load(open(tp))
                traffic = tj.get("k_frame_w_dram_bytes_per_launch")
                traffic_src = "static: " + tj.get("source", "ncu --set full capture kept in profiles/traffic.json")
            except Exception:
                traffic = None
        d2h = n * NF * CHANNELS * 4
        line = {
            "metric": "concurrent_realtime_48k_streams_decoded", "value": value, "unit": "streams",
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": 1e3 * t_value / K,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32+f32", "data": "synthetic",
            "config": workload_config(n, args.transient_permille, args.bitstream),
            "detail": {
                "cache": f"inputs larger than L2: {total} distinct packet sets resident in HBM, each read once; per 4096 streams "
                         "the decoder's PCM ring is 94 MB and every step writes 31.5 MB of new PCM into it",
                "per_kernel_ms": {"k_synth_rangedec": k0_ms, "k_frame_w": k1_ms, "k_synth_expand (unfused variant only)": k2_ms,
                                  "note": "second pass of the same steps, stages in order on one stream with cudaEvents around "
                                          "each; in the measured run the range decode of up to 8 later steps overlaps the frame kernel of step n"},
                "host_enqueue_ms_per_step": host_enqueue_ms,
                "peak_source": peak_src, "e2e_checksum": checksum, "rank_cpus": cpus,
            },
            "e2e": {"value": e2e, "unit": "streams", "h2d_bytes_per_step": step_bytes + 4 * 4 * n,
                    "d2h_bytes_per_step": d2h, "ms_per_step": 1e3 * t_e2e / K,
                    "pcie_peak_gbs": pcie_gbs, "pcie_frac": (d2h / (t_e2e / K) / 1e9) / pcie_gbs,
                    "pcie_note": f"pcie_peak_gbs = plain pinned D2H copies of {d2h} bytes, {world} rank(s) at once, per GPU (slowest rank); "
                                 "pcie_frac = this rank's PCM download rate inside the e2e loop / that ceiling"},
            "e2e_i16": {"value": world * n * K16 / t_e2e16 * FRAME_S, "unit": "streams", "steps": K16,
                        "d2h_bytes_per_step": n * NF * CHANNELS * 2, "ms_per_step": 1e3 * t_e2e16 / K16,
                        "note": "extra: the same host-buffer loop through opn_batch_decode_i16 (Decoder::decode::<i16>: "
                                "soft clip and sample conversion on the device); not the headline"},
            "e2e_pageable": {"value": world * n * KP / t_pg * FRAME_S, "unit": "streams", "steps": KP, "ms_per_step": 1e3 * t_pg / KP,
                             "note": "extra: pageable caller buffers (plain numpy arrays = what a Rust slice is), one synchronous call per step; "
                                     "the headline e2e uses pinned buffers (opn_host_alloc / opn_host_register) and two calls in flight"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": "k_frame_w<3,2,true> (PVQ expansion + IMDCT/TDAC + comb post-filter + PCM store)",
                         "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                         "algorithmic_bytes_per_launch": algo_bytes,
                         "bytes_note": f"{ch_frames} channel-frames x 4*(2*960+120) B (coefficients + carry in, PCM + carry out, SURVEY 8d) "
                                       f"+ 4 B x {hist_samples:.0f} comb history samples (sum of max(T0,T1)+2 over the channel-frames the "
                                       "post-filter ran on, counted by the kernel)"},
            "cpu_baseline": cpu,
            "clocks": clocks,
        }
        emit(line)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
