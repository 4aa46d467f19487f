"""opus-native_b200 -- host-side Python mirror of the reference crate's decode interface
(`Decoder`, `DecoderConfiguration`, `query_packet_*`, `parse_packet`; src/decoder.rs, src/lib.rs)
on top of the C ABI of libopusb200.so (include/opusb200.h).

Python is only plumbing here: it marshals numpy / torch buffers into the C ABI.  All decode work
happens in the hand-written sm_100a kernels inside the shared library; if the library is missing
or no B200-class device is usable every decode call raises -- there is no CPU fallback.
"""
from ._capi import (  # noqa: F401
    OpusError, lib, library_path, build_library,
    query_packet_bandwidth, query_packet_channel_count, query_packet_frame_count,
    query_packet_samples_per_frame, query_packet_sample_count, query_packet_codec_mode, parse_packet,
    DecoderConfiguration, Decoder, BatchDecoder, HostBuffer, host_register, host_unregister,
    op_rangedec_script, op_imdct_tdac, op_comb_filter_inplace, op_comb_filter, op_pcm_soft_clip, op_bitexact_trig, op_smooth_fade,
    op_synth_symbols, synth_packet, synth_fill, enc_run_script, op_celt2_symbols, celt2_packet, celt2_fill, CELT2_SIDE_DTYPE,
    silk_fill, op_silk_frames, SILK_SIDE_DTYPE, SILK_MAX_FRAME, BITSTREAM_SYNTH_SILK_1, FLAG_SILK_FRAMES, FLAG_DECODE_FEC, FLAG_MIXED_MODES,
    OP_DTYPE, OUT_DTYPE, SIDE_DTYPE,
    OP_UINT, OP_BITS, OP_BIT_LOGP, OP_ICDF, OP_LAPLACE, OP_BIT_VIA_DECODE, OP_BIT_VIA_DECODE_BIN,
    OP_PULSES, OP_SHRINK, OP_TELL, OP_PULSES_EVENTS, FLAG_DEVICE_PTRS, FLAG_NO_PCM_COPY, FLAG_INPUTS_READY, FLAG_SUBMIT_ONLY, FLAG_MIXED_FRAMES,
    BITSTREAM_OPUS, BITSTREAM_SYNTH_CELT_1, BITSTREAM_SYNTH_CELT_2,
    SAMPLE_F32, SAMPLE_I16, SAMPLE_I32, SAMPLE_U16, SAMPLE_U32, SAMPLE_F64, SAMPLE_FORMAT_OF,
)
from .sharding import shard_range  # noqa: F401

__all__ = [n for n in dir() if not n.startswith("_")]
