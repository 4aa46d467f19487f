"""Mixed-mode device-resident steps (OPN_FLAG_MIXED_MODES) at the shape of BASELINE configs[4]: per GPU, stereo streams of which
a share is in SILK (NB/MB/WB, 10 or 20 ms) and the rest in CELT (2.5/5/10/20 ms at 10/10/30/50 %, 10 % transient frames), a
share switching codec every step and a share of packets lost.  Timing and metric follow bench.py --mix: device events around
K back-to-back steps, audio seconds decoded per wall-clock second = concurrent realtime streams.  One JSON line.

Two yardsticks run in the same process:
  host_path: the same packets through the host-buffer call (page-locked buffers), what such traffic takes without this step;
  split:     the CELT streams of the first step as one OPN_FLAG_MIXED_FRAMES batch and the SILK streams as one
             OPN_FLAG_SILK_FRAMES batch at 20 ms, back to back, no switches: an estimate of the least the traffic could cost.

    python tools/bench_mixed_modes.py --streams 32768 --steps 200 --warmup 20
    torchrun --nproc_per_node 8 tools/bench_mixed_modes.py ..."""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import bench  # noqa: E402
from mixed_modes_oracle import mixed_mode_traffic  # noqa: E402  (the traffic the tests check, tests/test_gpu_mixed_modes.py)

CHANNELS = 2
CAP = 960


def gpu_name_and_power(index):
    import torch
    name = torch.cuda.get_device_name(index)
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unknown"
    return name, out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--streams", type=int, default=32768, help="streams per GPU")
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--silk-share", type=float, default=0.5)
    ap.add_argument("--switch-share", type=float, default=0.02, help="share of streams that switch codec per step")
    ap.add_argument("--loss-share", type=float, default=0.02)
    ap.add_argument("--transient-permille", type=int, default=100)
    args = ap.parse_args()
    import torch
    import opus_native_b200 as opn

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench_mixed_modes.py needs a CUDA device: libopusb200 has no CPU fallback")
    bench.pin_rank_to_cpus(local, world)
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
    cores = bench.cpu_threads()
    lo, _ = opn.shard_range(n * world, rank, world)

    def celt_fill(first, nn, frame, lm, ch, nb, tp):
        return opn.synth_fill(lo + first, nn, frame, 1, lm, ch, nb, tp, n_threads=cores)[0]

    def silk_fill(first, nn, frame, bw, ms, ch, nb):
        return opn.silk_fill(lo + first, nn, frame, 1, bw, ms, ch, nb, n_threads=cores)[0]

    rnd = np.random.default_rng(4321 + rank)
    packets, lens = mixed_mode_traffic(n, total, CHANNELS, rnd, celt_fill, silk_fill, seed=17, silk_share=args.silk_share,
                                       switch=args.switch_share, loss=args.loss_share, plc=0.0, first_loss=0.0,
                                       transient_permille=args.transient_permille)
    stride = packets.shape[2]

    def timed_loop(dec, step, k0, k1, host_s):
        stream = torch.cuda.ExternalStream(dec.cuda_stream, device=dev)
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

    # ---- the mixed-mode step
    dec = opn.BatchDecoder(n, opn.DecoderConfiguration(48000, CHANNELS, 0), device=local,
                           bitstream=opn.BITSTREAM_SYNTH_CELT_1 | opn.BITSTREAM_SYNTH_SILK_1)
    d_arena = torch.from_numpy(packets.reshape(-1)).to(dev)
    d_off = (torch.arange(n, dtype=torch.int64, device=dev) * stride).to(torch.int32)
    d_len = torch.from_numpy(lens.astype(np.int32)).to(dev)
    d_res = torch.zeros((total, n), dtype=torch.int32, device=dev)
    flags = opn.FLAG_DEVICE_PTRS | opn.FLAG_NO_PCM_COPY | opn.FLAG_INPUTS_READY | opn.FLAG_MIXED_MODES

    def step(f):
        dec.decode_float_ptrs(d_arena.data_ptr() + f * n * stride, d_off.data_ptr(), d_len[f].data_ptr(), None, 0, CAP,
                              d_res[f].data_ptr(), flags)

    for f in range(W):
        step(f)
    dec.synchronize()
    dec.stats(reset=True)
    host_s = [0.0]
    t = timed_loop(dec, step, W, total, host_s)
    res = d_res.cpu().numpy()
    assert (res[W:] > 0).all(), "decode reported errors"
    audio_s = float(res[W:].astype(np.int64).sum()) / 48000.0
    launches = dec.stats(reset=True)["launches"]
    dec.reset()
    dec.enable_timing(True)
    for f in range(W):
        step(f)
    dec.stats(reset=True)
    timed_loop(dec, step, W, total, [0.0])
    st = dec.stats(reset=True)
    dec.enable_timing(False)
    del dec

    # ---- yardstick 1: the host-buffer call on the same packets
    hdec = opn.BatchDecoder(n, opn.DecoderConfiguration(48000, CHANNELS, 0), device=local,
                            bitstream=opn.BITSTREAM_SYNTH_CELT_1 | opn.BITSTREAM_SYNTH_SILK_1)
    h_arena = opn.HostBuffer(packets.shape, np.uint8)
    h_arena.array[:] = packets
    h_pcm = opn.HostBuffer((n, CAP * CHANNELS), np.float32)
    h_off = (np.arange(n) * stride).astype(np.uint32)
    h_lens = lens.astype(np.uint32)
    hk = min(K, 40)
    for f in range(min(W, 5)):
        hdec.decode_float(h_arena.array[f].reshape(-1), h_off, h_lens[f], h_pcm.array, CAP)
    barrier()
    h0 = time.perf_counter()
    for f in range(W, W + hk):
        hdec.decode_float(h_arena.array[f].reshape(-1), h_off, h_lens[f], h_pcm.array, CAP)
    barrier()
    t_host = time.perf_counter() - h0
    audio_host = float(res[W:W + hk].astype(np.int64).sum()) / 48000.0
    del hdec

    # ---- yardstick 2: CELT half as a mixed-frame batch + SILK half as a SILK-frames batch (20 ms), no switches
    silk0 = (packets[0, :, 0] & 0x80) == 0
    nc, ns = int((~silk0).sum()), int(silk0.sum())
    srnd = np.random.default_rng(99 + rank)
    lm_of = srnd.choice(4, size=(total, nc), p=[0.1, 0.1, 0.3, 0.5])
    cbytes = {0: 64, 1: 80, 2: 110, 3: 160}
    c_pk = np.zeros((total, nc, 160), np.uint8)
    c_len = np.zeros((total, nc), np.int32)
    for f in range(total):
        for lm in range(4):
            ids = np.nonzero(lm_of[f] == lm)[0]
            if len(ids):
                c_pk[f, ids, :cbytes[lm]] = opn.synth_fill(lo + 7 * lm, len(ids), f, 1, lm, CHANNELS, cbytes[lm], args.transient_permille, n_threads=cores)[0]
                c_len[f, ids] = cbytes[lm]
    s_pk = np.zeros((total, ns, 120 * CHANNELS), np.uint8)
    bw = srnd.integers(0, 3, ns)
    for b in range(3):
        ids = np.nonzero(bw == b)[0]
        if len(ids):
            s_pk[:, ids] = opn.silk_fill(lo + 300 + b, len(ids), 0, total, b, 20, CHANNELS, 120 * CHANNELS, n_threads=cores)
    s_len = np.full((total, ns), 120 * CHANNELS, np.int32)
    for arr in (c_len, s_len):
        arr[srnd.random(arr.shape) < args.loss_share] = 0
    cdec = opn.BatchDecoder(nc, opn.DecoderConfiguration(48000, CHANNELS, 0), device=local, bitstream=opn.BITSTREAM_SYNTH_CELT_1)
    sdec = opn.BatchDecoder(ns, opn.DecoderConfiguration(48000, CHANNELS, 0), device=local,
                            bitstream=opn.BITSTREAM_SYNTH_CELT_1 | opn.BITSTREAM_SYNTH_SILK_1)
    dc = (torch.from_numpy(c_pk.reshape(-1)).to(dev), (torch.arange(nc, dtype=torch.int64, device=dev) * 160).to(torch.int32),
          torch.from_numpy(c_len).to(dev), torch.zeros(nc, dtype=torch.int32, device=dev))
    sp = 120 * CHANNELS
    ds = (torch.from_numpy(s_pk.reshape(-1)).to(dev), (torch.arange(ns, dtype=torch.int64, device=dev) * sp).to(torch.int32),
          torch.from_numpy(s_len).to(dev), torch.zeros(ns, dtype=torch.int32, device=dev))
    base = opn.FLAG_DEVICE_PTRS | opn.FLAG_NO_PCM_COPY | opn.FLAG_INPUTS_READY

    def split_step(f):
        cdec.decode_float_ptrs(dc[0].data_ptr() + f * nc * 160, dc[1].data_ptr(), dc[2][f].data_ptr(), None, 0, CAP, dc[3].data_ptr(),
                               base | opn.FLAG_MIXED_FRAMES)
        sdec.decode_float_ptrs(ds[0].data_ptr() + f * ns * sp, ds[1].data_ptr(), ds[2][f].data_ptr(), None, 0, 960, ds[3].data_ptr(),
                               base | opn.FLAG_SILK_FRAMES)

    for f in range(W):
        split_step(f)
    cdec.synchronize()
    sdec.synchronize()
    barrier()
    stream = torch.cuda.ExternalStream(cdec.cuda_stream, device=dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        e0.record()
        for f in range(W, total):
            split_step(f)
        cdec.join()
        sdec.join()
        ev = torch.cuda.Event()
        ev.record(torch.cuda.ExternalStream(sdec.cuda_stream, device=dev))
        stream.wait_event(ev)
        e1.record()
    cdec.synchronize()
    sdec.synchronize()
    t_split = e0.elapsed_time(e1) * 1e-3
    audio_split = (float((120 << lm_of[W:]).sum()) + 960.0 * ns * K) / 48000.0

    if dist is not None:
        v = torch.tensor([t, t_host, t_split], dtype=torch.float64, device=dev)
        dist.all_reduce(v, op=dist.ReduceOp.MAX)
        t, t_host, t_split = (float(x) for x in v.tolist())
        a = torch.tensor([audio_s, audio_host, audio_split], dtype=torch.float64, device=dev)
        dist.all_reduce(a, op=dist.ReduceOp.SUM)
        audio_s, audio_host, audio_split = (float(x) for x in a.tolist())
    name, power = gpu_name_and_power(local)
    if rank == 0:
        bench.emit({
            "metric": "concurrent_realtime_48k_streams_decoded", "value": audio_s / t, "unit": "streams", "n_gpus": world, "steps": K,
            "warmup": W, "us_per_step": 1e6 * t / K, "higher_is_better": True, "gpu": name, "power_limit": power,
            "config": {"workload": f"{n} stereo streams per GPU, {100 * args.silk_share:.0f} % SILK (NB/MB/WB, 10/20 ms), CELT 2.5/5/10/20 ms "
                                   f"at 10/10/30/50 % ({args.transient_permille / 10:.0f} % transient), {100 * args.switch_share:.0f} % switch codec "
                                   f"per step, {100 * args.loss_share:.0f} % lost; device-resident, OPN_FLAG_MIXED_MODES",
                       "streams_per_gpu": n, "silk_share": args.silk_share, "switch_share": args.switch_share, "loss_share": args.loss_share},
            "launches_per_step": [x / K for x in launches], "host_enqueue_us_per_step": 1e6 * host_s[0] / K,
            "stage_ms_per_step_timed_pass": {"range_decodes": st["ms"][0] / K, "frame_kernels_and_switches": st["ms"][1] / K},
            "host_path": {"value": audio_host / t_host, "us_per_step": 1e6 * t_host / hk, "steps": hk},
            "split": {"value": audio_split / t_split, "us_per_step": 1e6 * t_split / K, "celt_streams": nc, "silk_streams_20ms": ns},
        })
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
