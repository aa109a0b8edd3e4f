"""B200-native JPEG encode path behind the jpeg-encoder (Rust crate) API.

Package contents: csrc/ (CUDA kernels + C ABI + host planner), encoder.py (ctypes mirror of the
reference's `Encoder`), build.py (nvcc build of libjpegenc_b200.so). No CPU fallback exists.
"""
from .encoder import (ColorType, Device, Encoder, EncodingError, JpegColorType, PixelDensity, PixelDensityUnit,  # noqa: F401
                      QuantizationTableType, SampleType, SamplingFactor, default_device, load_library, sample_scale_offset)
