"""canny_edge_b200 — B200-native (sm_100a) Canny edge hot path behind the reference's stage API.

Layout:
  csrc/      hand-written CUDA kernels + the C ABI (include/canny_b200.h) -> libcanny_b200.so
  _lib.py    ctypes binding of that ABI (fails loudly when the library is missing)
  api.py     host-side mirror of the reference interface (src/cuda.h / src/utils.h names)
  torch_api.py  CUDA uint8 tensors in and out, any row-contiguous view (crops, channels, padded rows) without a copy
  sharded.py frame- and row-band sharding across GPUs (torch.distributed over NCCL as plumbing)
  cli.py     file front end with the reference CLI's arguments (src/main.cpp reads a webcam; this reads image files)
  build.py   in-tree nvcc build
"""
from ._lib import CannyB200Error, LIB_PATH, load  # noqa: F401
from .api import (  # noqa: F401
    EDGE, NOEDGE, PI, Context, calculateXYGradient, canny_batch_device_bgr_ptr, canny_batch_device_bgr_strided_ptr, canny_batch_device_ptr,
    canny_batch_device_strided_ptr, canny_batch_host, canny_frames_device_ptr, createGaussianKernel, cv_canny_device_strided_ptr, cv_canny_frames_device_ptr,
    cv_gaussian_canny_device_strided_ptr, cv_gaussian_canny_frames_device_ptr, cv_gaussian_kernel, cuda_canny, cuda_canny_bgr, cuda_gaussian, cuda_hysteresis,
    cuda_nonmaixmal_suppression, cuda_sobel, synth_host, synth_rows_host,
)
from . import torch_api  # noqa: F401  (torch is imported inside its functions)
