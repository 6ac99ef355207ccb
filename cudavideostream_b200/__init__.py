"""cudavideostream_b200 -- B200-native (sm_100a) replacement for the per-pixel hot path of
MatteoBattilana/CUDAVideoStream's server: thresholded frame difference with negative feedback, ordered
compaction into the (index, value) payload, and the display-filter chain.

The product is libcvs_b200.so (hand-written CUDA kernels behind the C ABI of include/cvs_b200.h, plus a
drop-in diff::cuda::CUDACore for the reference's C++ server).  This Python package is a thin ctypes view
of that ABI for tests and benchmarks.  There is no CPU fallback: importing works anywhere, every compute
call needs the built library and an sm_100 GPU and fails loudly otherwise.
"""
from .api import (CVSError, CUDACore, Stream, alloc_host, device_count, library_path, load_library,  # noqa: F401
                  MODE_NONE, MODE_HEAT_MAP, MODE_RED_BLACK, MODE_RED_OVERLAP, MODE_GRAY_WEIGHTED,
                  MODE_BINARIZE, MODE_GRAY_AVERAGE, MODE_BINARIZE_AVERAGE, MAX_BATCH, run_batch_device, submit_io_batch)
from . import filters, sharding, synth, wire  # noqa: F401

__all__ = ["CVSError", "CUDACore", "Stream", "alloc_host", "device_count", "library_path", "load_library",
           "run_batch_device", "submit_io_batch", "filters", "sharding", "synth", "wire"]
