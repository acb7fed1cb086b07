"""B200-native RTjpeg decoder (and converters, encoder) behind gmerlin-avdecoder's own interfaces.

The product is the C-ABI library built from ``csrc/`` (CUDA kernels for sm_100a,
batch context, ``RTjpeg.h``-compatible shim, ``'RTJ0'`` bgav plugin).  This
Python package is only the binding that tests and ``bench.py`` drive it through:

* :mod:`capi`   -- ctypes mirror of ``include/rtjpeg_b200.h``
* :mod:`device` -- torch-backed device buffers for the device-resident entry point

The library also carries a NuppelVideo container reader (``rtjnuv_*``) that rewraps the RTjpeg
frames of a ``.nuv`` file as ``'RTJ0'`` packets for the decoder.

The directory name carries a hyphen (it is the reference's name); import it as
``gmerlin_avdecoder_b200`` through the shim module at the repository root.
"""
from .capi import (  # noqa: F401
    BatchContext, BatchInfo, RTjpeg, RTjpegError, SeqEncoder, State, Timing,
    FRAME_DESC_DTYPE, HOST_IN_PINNED, HOST_OUT_PINNED, LIB_PATH, PLUGIN_PATH, STREAM_SLACK_BYTES,
    TABLE_CUSTOM, TABLE_ZERO, PIPELINE_AUTO, PIPELINE_SERIAL, PIPELINE_SLICED, CONV_BPP, CONVERTERS, NuvHeader, build_library, load_library, nuv_extract_rtj0, nuv_open, nuv_packets, nuv_probe,
    encode_bound, plan, plan_sequences, raw_tables_for_quality, select_frames, split_shards, split_shards_lead, tables_for_quality, tables_from_raw,
)
