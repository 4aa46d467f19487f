"""The timed pass (opn_batch_enable_timing) against the pipelined one.  With timing on, every launch of a step sits between two
events on the batch stream, so the benchmark can attribute time to each kernel; the decode itself must not change.  Each case
decodes the same device-resident steps, enqueued back to back, with two identically configured batches, one timed and one
not, and asserts bit-identical PCM, per-stream results and final ranges, and the launches per step that each mode makes:
[range decodes, frame-kernel launches, bucketing kernels of a mixed-frame step]."""
import numpy as np
import pytest

import opus_native_b200 as opn

pytestmark = pytest.mark.gpu
NSTEPS = 4
SILK = opn.BITSTREAM_SYNTH_CELT_1 | opn.BITSTREAM_SYNTH_SILK_1


def _celt_steps(ns, channels, rnd):
    pkt_bytes = 160
    packets = opn.synth_fill(int(rnd.integers(1 << 20)), ns, 0, NSTEPS, 3, channels, pkt_bytes, transient_permille=100)
    return packets, np.full((NSTEPS, ns), pkt_bytes, np.uint32), 960, opn.BITSTREAM_SYNTH_CELT_1, 0


def _silk_steps(ns, channels, rnd):
    nb = 96 * channels
    packets = opn.silk_fill(int(rnd.integers(1 << 20)), ns, 0, NSTEPS, 2, 20, channels, nb)  # wideband, 20 ms
    lens = np.full((NSTEPS, ns), nb, np.uint32)
    lens[2, ::9] = 0
    return packets, lens, 960, SILK, opn.FLAG_SILK_FRAMES


def _mixed_steps(ns, channels, rnd):
    """every stream picks a frame size per step (2.5/5/10/20 ms); 3 % of the packets after the first step are lost"""
    stride, pkt_bytes = 160, {0: 64, 1: 80, 2: 110, 3: 160}
    packets = np.zeros((NSTEPS, ns, stride), np.uint8)
    lens = np.zeros((NSTEPS, ns), np.uint32)
    for f in range(NSTEPS):
        lm_of = rnd.choice([0, 1, 2, 3], size=ns, p=[0.1, 0.1, 0.3, 0.5])
        for lm in range(4):
            ids = np.nonzero(lm_of == lm)[0]
            if len(ids):
                packets[f, ids, :pkt_bytes[lm]] = opn.synth_fill(700 + lm, len(ids), f, 1, lm, channels, pkt_bytes[lm], transient_permille=100)[0]
                lens[f, ids] = pkt_bytes[lm]
        if f > 0:
            lens[f, rnd.random(ns) < 0.03] = 0
    return packets, lens, 960, opn.BITSTREAM_SYNTH_CELT_1, opn.FLAG_MIXED_FRAMES


def _decode(packets, lens, cap, bitstream, flags, channels, timing):
    torch = pytest.importorskip("torch")
    nsteps, ns, stride = packets.shape
    dev = torch.device("cuda:0")
    d_arena = torch.from_numpy(packets.reshape(-1).copy()).to(dev)
    d_off = torch.arange(ns, dtype=torch.int32, device=dev) * stride
    d_len = torch.from_numpy(lens.astype(np.int32)).to(dev)
    d_pcm = torch.full((nsteps, ns, cap * channels), 7.0, dtype=torch.float32, device=dev)
    d_res = torch.full((nsteps, ns), -99, dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    dec = opn.BatchDecoder(ns, opn.DecoderConfiguration(48000, channels, 0), bitstream=bitstream)
    dec.enable_timing(timing)
    flags |= opn.FLAG_DEVICE_PTRS | opn.FLAG_INPUTS_READY
    for f in range(nsteps):
        dec.decode_float_ptrs(d_arena.data_ptr() + f * ns * stride, d_off.data_ptr(), d_len[f].data_ptr(), d_pcm[f].data_ptr(),
                              cap * channels, cap, d_res[f].data_ptr(), flags)
    dec.join()
    dec.synchronize()
    return d_pcm.cpu().numpy(), d_res.cpu().numpy(), dec.final_ranges(), dec.stats()["launches"]


# (steps, streams, channels, launches per step untimed, launches per step timed).  2048 streams and more run the frame kernel
# as three concurrent launches; the SILK timed pass launches it once.
CASES = {
    "celt-4096": (_celt_steps, 4096, 2, [1, 3, 0], [1, 3, 0]),
    "silk-2300": (_silk_steps, 2300, 1, [1, 3, 0], [1, 1, 0]),
    "mixed-2300": (_mixed_steps, 2300, 2, [1, 3, 2], [1, 3, 2]),
    "celt-300": (_celt_steps, 300, 2, [1, 1, 0], [1, 1, 0]),
    "silk-300": (_silk_steps, 300, 1, [1, 1, 0], [1, 1, 0]),
    "mixed-300": (_mixed_steps, 300, 2, [1, 1, 2], [1, 1, 2]),
}


@pytest.mark.parametrize("case", list(CASES))
def test_timed_pass_decodes_what_the_pipelined_pass_decodes(case):
    steps, ns, channels, want_untimed, want_timed = CASES[case]
    packets, lens, cap, bitstream, flags = steps(ns, channels, np.random.default_rng(ns))
    pcm0, res0, rng0, launches0 = _decode(packets, lens, cap, bitstream, flags, channels, timing=False)
    pcm1, res1, rng1, launches1 = _decode(packets, lens, cap, bitstream, flags, channels, timing=True)
    assert np.all(res0 > 0) and np.abs(pcm0).max() > 0.01
    assert np.array_equal(res1, res0)
    for f in range(NSTEPS):
        assert np.array_equal(pcm1[f].view(np.uint32), pcm0[f].view(np.uint32)), f
    assert np.array_equal(rng1, rng0)
    assert launches0 == [NSTEPS * k for k in want_untimed]
    assert launches1 == [NSTEPS * k for k in want_timed]
