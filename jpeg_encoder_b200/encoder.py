"""Host-side mirror of the reference crate's public encode API over the C ABI (ctypes).

Same names, argument meaning and error behaviour as `jpeg_encoder::Encoder`
(/root/reference/src/encoder.rs:213-515): `Encoder(quality)`, the setters, `encode(data, w, h,
color_type)`. The reference writes into a `W: JfifWrite`; here `encode` returns the bytes, and
`encode_to(writer, ...)` calls `writer.write(bytes)` like the blanket `std::io::Write` impl
(src/writer.rs:99-106).

There is no CPU path: if the CUDA library is missing or no B200 is present, construction of the
device context raises.
"""
import ctypes as C
import enum
import os

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_PKG, "libjpegenc_b200.so")


class ColorType(enum.IntEnum):
    """src/encoder.rs:72-99"""
    Luma = 0
    Rgb = 1
    Rgba = 2
    Bgr = 3
    Bgra = 4
    Ycbcr = 5
    Cmyk = 6
    CmykAsYcck = 7
    Ycck = 8

    def get_bytes_per_pixel(self):
        return (1, 3, 4, 3, 4, 3, 4, 4, 4)[int(self)]


class JpegColorType(enum.IntEnum):
    """src/encoder.rs:21-65 (colour type of the encoded file; what an ImageBuffer reports)"""
    Luma = 0
    Ycbcr = 1
    Cmyk = 2
    Ycck = 3

    def get_num_components(self):
        return (1, 3, 4, 4)[int(self)]

    def as_color_type(self):
        return (ColorType.Luma, ColorType.Ycbcr, ColorType.Cmyk, ColorType.Ycck)[int(self)]


class SamplingFactor(enum.IntEnum):
    """src/encoder.rs:120-153 ((h << 4) | v; R_* aliases carry bit 0x80)"""
    F_1_1 = 1 << 4 | 1
    F_2_1 = 2 << 4 | 1
    F_1_2 = 1 << 4 | 2
    F_2_2 = 2 << 4 | 2
    F_4_1 = 4 << 4 | 1
    F_4_2 = 4 << 4 | 2
    F_1_4 = 1 << 4 | 4
    F_2_4 = 2 << 4 | 4
    R_4_4_4 = 0x80 | 1 << 4 | 1
    R_4_4_0 = 0x80 | 1 << 4 | 2
    R_4_4_1 = 0x80 | 1 << 4 | 4
    R_4_2_2 = 0x80 | 2 << 4 | 1
    R_4_2_0 = 0x80 | 2 << 4 | 2
    R_4_2_1 = 0x80 | 2 << 4 | 4
    R_4_1_1 = 0x80 | 4 << 4 | 1
    R_4_1_0 = 0x80 | 4 << 4 | 2

    @staticmethod
    def from_factors(horizontal, vertical):
        """src/encoder.rs:157-171"""
        for f in (SamplingFactor.F_1_1, SamplingFactor.F_1_2, SamplingFactor.F_1_4, SamplingFactor.F_2_1,
                  SamplingFactor.F_2_2, SamplingFactor.F_2_4, SamplingFactor.F_4_1, SamplingFactor.F_4_2):
            if f.get_sampling_factors() == (horizontal, vertical):
                return f
        return None

    def get_sampling_factors(self):
        return ((int(self) >> 4) & 0x07, int(self) & 0xF)


class QuantizationTableType(enum.IntEnum):
    """src/quantization.rs:8-40; Custom is expressed by passing a sequence of 64 u16 instead."""
    Default = 0
    Flat = 1
    CustomMsSsim = 2
    CustomPsnrHvs = 3
    ImageMagick = 4
    KleinSilversteinCarney = 5
    DentalXRays = 6
    VisualDetectionModel = 7
    ImprovedDetectionModel = 8


class PixelDensityUnit(enum.IntEnum):
    """src/writer.rs:47-59"""
    PixelAspectRatio = 0
    Inches = 1
    Centimeters = 2


class PixelDensity:
    """src/writer.rs:16-45"""

    def __init__(self, density=(1, 1), unit=PixelDensityUnit.PixelAspectRatio):
        self.density = tuple(density)
        self.unit = PixelDensityUnit(unit)

    @staticmethod
    def dpi(density):
        return PixelDensity((density, density), PixelDensityUnit.Inches)

    def __eq__(self, o):
        return isinstance(o, PixelDensity) and self.density == o.density and self.unit == o.unit


class EncodingError(Exception):
    """src/error.rs:6-28; `.kind` names the variant."""
    KINDS = {1: "BadImageData", 2: "ZeroImageDimensions", 3: "InvalidAppSegment", 4: "AppSegmentTooLarge",
             5: "BadParams", 6: "Write", 7: "OutOfMemory", 8: "Cuda", 9: "Huffman", 10: "IccTooLarge"}

    def __init__(self, code, message=""):
        self.code = code
        self.kind = self.KINDS.get(code, "Unknown")
        super().__init__("%s: %s" % (self.kind, message) if message else self.kind)


class _App(C.Structure):
    _fields_ = [("nr", C.c_uint8), ("data", C.POINTER(C.c_uint8)), ("len", C.c_uint32)]


class _Params(C.Structure):
    _fields_ = [
        ("width", C.c_uint16), ("height", C.c_uint16),
        ("color_type", C.c_uint8), ("quality", C.c_uint8), ("sampling", C.c_uint8),
        ("qtable_kind", C.c_uint8 * 2),
        ("qtable_custom", (C.c_uint16 * 64) * 2),
        ("progressive_scans", C.c_uint8), ("optimize_huffman", C.c_uint8),
        ("restart_interval", C.c_uint16),
        ("density_unit", C.c_uint8), ("density_x", C.c_uint16), ("density_y", C.c_uint16),
        ("n_app", C.c_uint32), ("apps", C.POINTER(_App)),
    ]


class _CoefLayout(C.Structure):
    _fields_ = [("n_components", C.c_uint32), ("blocks_w", C.c_uint32 * 4), ("blocks_h", C.c_uint32 * 4),
                ("true_w", C.c_uint32 * 4), ("true_h", C.c_uint32 * 4), ("block_offset", C.c_uint64 * 4),
                ("blocks_per_image", C.c_uint64), ("mcu_order", C.c_uint32), ("mcu_cols", C.c_uint32), ("mcu_rows", C.c_uint32),
                ("blocks_per_mcu", C.c_uint32), ("slot_base", C.c_uint32 * 4), ("comp_h", C.c_uint32 * 4), ("comp_v", C.c_uint32 * 4)]


class _Strip(C.Structure):
    _fields_ = [("strip_index", C.c_uint32), ("n_strips", C.c_uint32), ("first_row", C.c_uint16), ("rows", C.c_uint16),
                ("full_height", C.c_uint16)]


class _DeviceImages(C.Structure):
    _fields_ = [("data", C.c_void_p), ("image_stride", C.c_uint64), ("row_stride", C.c_uint64), ("plane_stride", C.c_uint64)]


N_STAGES = 7
HIST_WORDS = 2 * 2 * 257  # JPGB_HIST_WORDS
STAGE_NAMES = ("colour_dct_quant", "histogram_tables", "code_chunks_scans", "place_chunks", "stuff_scatter", "h2d", "d2h")

_lib = None


def load_library():
    """Load libjpegenc_b200.so (built in-tree by jpeg_encoder_b200.build). Fails loudly if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise RuntimeError("CUDA library %s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback)" % _LIB_PATH)
    l = C.CDLL(_LIB_PATH)
    vp, u8p = C.c_void_p, C.POINTER(C.c_uint8)
    l.jpgb_params_default.argtypes = [C.POINTER(_Params), C.c_uint8]
    l.jpgb_params_default.restype = None
    l.jpgb_encoder_create.argtypes = [C.c_int, vp, C.POINTER(vp)]
    l.jpgb_encoder_destroy.argtypes = [vp]
    l.jpgb_encoder_destroy.restype = None
    l.jpgb_last_error.argtypes = [vp]
    l.jpgb_last_error.restype = C.c_char_p
    l.jpgb_encode.argtypes = [vp, C.POINTER(_Params), vp, C.c_size_t, C.POINTER(u8p), C.POINTER(C.c_size_t)]
    l.jpgb_free.argtypes = [vp]
    l.jpgb_free.restype = None
    l.jpgb_encode_to_sink.argtypes = [vp, C.POINTER(_Params), vp, C.c_size_t, vp, vp]
    l.jpgb_encode_batch.argtypes = [vp, C.POINTER(_Params), C.POINTER(vp), C.c_size_t, C.c_uint32,
                                    C.POINTER(u8p), C.POINTER(C.c_size_t)]
    l.jpgb_encode_planar.argtypes = [vp, C.POINTER(_Params), C.POINTER(vp), C.c_size_t, C.POINTER(u8p), C.POINTER(C.c_size_t)]
    l.jpgb_encode_planar_to_sink.argtypes = [vp, C.POINTER(_Params), C.POINTER(vp), C.c_size_t, vp, vp]
    l.jpgb_encode_batch_pinned.argtypes = [vp, C.POINTER(_Params), C.POINTER(vp), C.c_size_t, C.c_uint32,
                                           C.POINTER(vp), C.POINTER(C.c_uint64)]
    l.jpgb_encode_batch_device.argtypes = [vp, C.POINTER(_Params), vp, C.c_size_t, C.c_uint32,
                                           C.POINTER(vp), C.POINTER(C.c_uint64)]
    l.jpgb_encode_batch_device_strided.argtypes = [vp, C.POINTER(_Params), C.POINTER(_DeviceImages), C.c_uint32,
                                                   C.POINTER(vp), C.POINTER(C.c_uint64)]
    l.jpgb_encoder_wait_stream.argtypes = [vp, vp]
    l.jpgb_scan_count.argtypes = [C.POINTER(_Params), C.POINTER(C.c_uint32)]
    l.jpgb_plan_strips.argtypes = [C.POINTER(_Params), C.c_uint32, C.POINTER(_Strip), C.POINTER(C.c_uint32)]
    l.jpgb_encode_strip_device.argtypes = [vp, C.POINTER(_Params), C.POINTER(_Strip), vp, C.POINTER(vp), C.POINTER(C.c_uint64)]
    l.jpgb_encode_strip_device_optimized.argtypes = [vp, C.POINTER(_Params), C.POINTER(_Strip), vp, C.POINTER(C.c_uint32), C.POINTER(vp),
                                                     C.POINTER(C.c_uint64)]
    l.jpgb_strip_histogram_device.argtypes = [vp, C.POINTER(_Params), C.POINTER(_Strip), vp, C.POINTER(C.c_uint32), C.POINTER(C.c_int16)]
    l.jpgb_merge_strip_histograms.argtypes = [C.POINTER(_Params), C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_int16), C.POINTER(C.c_uint32)]
    l.jpgb_download.argtypes = [vp, vp, C.c_size_t, vp]
    l.jpgb_gather_target_create.argtypes = [vp, C.c_size_t, C.POINTER(vp), u8p]
    l.jpgb_gather_target_open.argtypes = [vp, u8p, C.POINTER(vp)]
    l.jpgb_gather_target_close.argtypes = [vp, vp, C.c_int]
    l.jpgb_last_piece_offsets_device.argtypes = [vp, C.POINTER(vp), C.POINTER(C.c_uint32)]
    l.jpgb_gather_place_pieces.argtypes = [vp, vp, C.c_size_t, vp, C.c_uint32, C.c_uint32, vp]
    l.jpgb_coef_layout_for.argtypes = [C.POINTER(_Params), C.POINTER(_CoefLayout)]
    l.jpgb_stage_a_device.argtypes = [vp, C.POINTER(_Params), vp, C.c_size_t, C.c_uint32, vp]
    l.jpgb_encoder_set_timing.argtypes = [vp, C.c_int]
    l.jpgb_encoder_set_timing.restype = None
    l.jpgb_encoder_last_timing.argtypes = [vp, C.POINTER(C.c_float)]
    l.jpgb_encoder_last_launch_count.argtypes = [vp]
    l.jpgb_encoder_last_launch_count.restype = C.c_uint32
    l.jpgb_build_header.argtypes = [C.POINTER(_Params), u8p, C.c_size_t, C.POINTER(C.c_size_t)]
    l.jpgb_optimized_huffman_table.argtypes = [C.POINTER(C.c_uint32), u8p, u8p, C.POINTER(C.c_uint32)]
    l.jpgb_optimized_huffman_tables_device.argtypes = [vp, C.POINTER(C.c_uint32), C.c_uint32, C.c_int, u8p, u8p, C.POINTER(C.c_uint32),
                                                       C.POINTER(C.c_uint32), C.POINTER(C.c_int)]
    l.jpgb_version.restype = C.c_char_p
    _lib = l
    return l


class Device:
    """One jpgb_encoder context (device + stream + scratch). Not thread-safe; reuse across calls."""

    def __init__(self, device=0, cuda_stream=None):
        self.lib = load_library()
        h = C.c_void_p()
        rc = self.lib.jpgb_encoder_create(device, C.c_void_p(cuda_stream) if cuda_stream else None, C.byref(h))
        if rc != 0:
            raise EncodingError(rc, "jpgb_encoder_create(device=%d) failed: no usable sm_100 GPU (no CPU fallback)" % device)
        self.handle = h
        self.device = device

    def close(self):
        if getattr(self, "handle", None):
            self.lib.jpgb_encoder_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def download(self, d_ptr, nbytes):
        """Copy nbytes of device memory (e.g. the files of encode_batch_device) into a bytes object."""
        buf = C.create_string_buffer(nbytes)
        rc = self.lib.jpgb_download(self.handle, C.c_void_p(d_ptr), nbytes, buf)
        if rc != 0:
            raise EncodingError(rc, self.last_error())
        return buf.raw

    def last_error(self):
        return self.lib.jpgb_last_error(self.handle).decode()

    def set_timing(self, enabled):
        self.lib.jpgb_encoder_set_timing(self.handle, 1 if enabled else 0)

    def last_timing(self):
        ms = (C.c_float * N_STAGES)()
        if self.lib.jpgb_encoder_last_timing(self.handle, ms) != 0:
            return None
        return dict(zip(STAGE_NAMES, list(ms)))

    def last_launch_count(self):
        return int(self.lib.jpgb_encoder_last_launch_count(self.handle))

    def wait_stream(self, stream):
        """Order this context's stream after the work queued so far on `stream` (a cudaStream_t as an int; 1 is the
        legacy default stream, 2 the per-thread one). The host does not block."""
        rc = self.lib.jpgb_encoder_wait_stream(self.handle, C.c_void_p(stream))
        if rc != 0:
            raise EncodingError(rc, self.last_error())


_default_devices = {}


def default_device(device=0):
    if device not in _default_devices:
        _default_devices[device] = Device(device)
    return _default_devices[device]


def _host_view(data):
    if isinstance(data, np.ndarray):
        a = np.ascontiguousarray(data)
        if a.dtype != np.uint8:
            a = a.astype(np.uint8)
        return a.reshape(-1)
    return np.frombuffer(data, dtype=np.uint8)


def _cuda_array_layout(iface, bpp, channels_first):
    """The jpgb_device_images of a `__cuda_array_interface__` dict holding uint8 images:
    (data, n, width, height, image_stride, row_stride, plane_stride). Shapes: (H, W, C) / (N, H, W, C), or with
    channels_first (C, H, W) / (N, C, H, W); C must be the colour type's bytes per pixel. Raises ValueError for a
    layout the encoder cannot read in place."""
    if iface.get("typestr") != "|u1":
        raise ValueError("uint8 images only (typestr '|u1'), got %r" % (iface.get("typestr"),))
    if iface.get("mask") is not None:
        raise ValueError("masked arrays are not supported")
    shape = tuple(int(d) for d in iface["shape"])
    if len(shape) not in (3, 4):
        raise ValueError("expected a 3-D (one image) or 4-D (batch) array, got shape %r" % (shape,))
    strides = iface.get("strides")
    if strides is None:  # C-contiguous
        strides, step = [], 1
        for d in reversed(shape):
            strides.insert(0, step)
            step *= d
    strides = tuple(int(x) for x in strides)
    names = ("c", "y", "x") if channels_first else ("y", "x", "c")
    if len(shape) == 4:
        names = ("n",) + names
    for name, st in zip(names, strides):
        if st < 0:
            raise ValueError("negative %s stride %d: make the array .contiguous() first" % (name, st))
    dim = dict(zip(names, shape))
    stride = dict(zip(names, strides))
    if dim["c"] != bpp:
        raise ValueError("the colour type takes %d channels, the array has %d" % (bpp, dim["c"]))
    if channels_first:
        if stride["x"] != 1:
            raise ValueError("x stride %d: channel-planar rows must be contiguous; make the array .contiguous() first" % stride["x"])
        plane_stride = stride["c"] if bpp > 1 else 0  # one plane is packed Luma
        if bpp > 1 and plane_stride == 0:
            raise ValueError("channel stride 0: planes at one address cannot be read; make the array .contiguous() first")
    else:
        if stride["c"] != 1:
            raise ValueError("channel stride %d: channels must be adjacent; make the array .contiguous() first" % stride["c"])
        if stride["x"] != bpp:
            raise ValueError("pixel stride %d: pixels must be %d bytes apart; make the array .contiguous() first" % (stride["x"], bpp))
        plane_stride = 0
    if dim["x"] > 65535 or dim["y"] > 65535:
        raise ValueError("image dimensions above 65535 (%d x %d)" % (dim["x"], dim["y"]))
    return (int(iface["data"][0]), dim.get("n", 1), dim["x"], dim["y"], stride.get("n", 0), stride["y"], plane_stride)


class Encoder:
    """jpeg_encoder::Encoder (src/encoder.rs:213-515)."""

    def __init__(self, quality, device=None):
        """Encoder::new(w, quality), :239-275."""
        self._quality = int(quality) & 0xFF
        self._density = PixelDensity()
        self._quantization_tables = [QuantizationTableType.Default, QuantizationTableType.Default]
        self._sampling_factor = SamplingFactor.F_2_2 if quality < 90 else SamplingFactor.F_1_1
        self._progressive_scans = None
        self._restart_interval = None
        self._optimize_huffman_table = False
        self._app_segments = []
        self._device = device

    # -- setters / getters, :280-364 --
    def set_density(self, density):
        self._density = density

    def density(self):
        return self._density

    def set_sampling_factor(self, sampling):
        self._sampling_factor = SamplingFactor(sampling)

    def sampling_factor(self):
        return self._sampling_factor

    def set_quantization_tables(self, luma, chroma):
        """Each table: a QuantizationTableType, or 64 u16 values in natural order (Custom)."""
        self._quantization_tables = [luma, chroma]

    def quantization_tables(self):
        return self._quantization_tables

    def set_progressive(self, progressive):
        self._progressive_scans = 4 if progressive else None

    def set_progressive_scans(self, scans):
        if not 2 <= scans <= 64:  # the reference asserts (:329-333)
            raise ValueError("Invalid number of scans: %d" % scans)
        self._progressive_scans = scans

    def progressive_scans(self):
        return self._progressive_scans

    def set_restart_interval(self, interval):
        self._restart_interval = None if interval == 0 else interval

    def restart_interval(self):
        return self._restart_interval

    def set_optimized_huffman_tables(self, optimize_huffman_table):
        self._optimize_huffman_table = bool(optimize_huffman_table)

    def optimized_huffman_tables(self):
        return self._optimize_huffman_table

    # -- APP segments, :366-435 --
    def add_app_segment(self, segment_nr, data):
        if segment_nr == 0 or segment_nr > 15:
            raise EncodingError(3, "Invalid app segment number: %d" % segment_nr)
        if len(data) > 65533:
            raise EncodingError(4, "App segment exceeds maximum allowed data length of 65533: %d" % len(data))
        self._app_segments.append((segment_nr, bytes(data)))

    def add_icc_profile(self, data):
        marker = b"ICC_PROFILE\0"
        max_chunk = 65535 - 2 - 12 - 2
        num_chunks = (len(data) + max_chunk - 1) // max_chunk
        if num_chunks >= 255:
            raise EncodingError(10, "ICC profile exceeds maximum allowed data length: %d" % len(data))
        for i in range(num_chunks):
            chunk = data[i * max_chunk:(i + 1) * max_chunk]
            self.add_app_segment(2, marker + bytes([i + 1, num_chunks]) + bytes(chunk))

    def add_exif_metadata(self, data):
        self.add_app_segment(1, b"Exif\0\0" + bytes(data))

    # -- the C-ABI parameter block --
    def _params(self, width, height, color_type):
        p = _Params()
        p.width, p.height = width, height
        p.color_type = int(color_type)
        p.quality = self._quality
        p.sampling = int(self._sampling_factor) & 0xFF
        for i, t in enumerate(self._quantization_tables):
            if isinstance(t, (QuantizationTableType, int)):
                p.qtable_kind[i] = int(t)
            else:
                vals = list(t)
                if len(vals) != 64:
                    raise ValueError("custom quantization table needs 64 values")
                p.qtable_kind[i] = 9
                for k in range(64):
                    p.qtable_custom[i][k] = int(vals[k]) & 0xFFFF
        p.progressive_scans = self._progressive_scans or 0
        p.optimize_huffman = 1 if self._optimize_huffman_table else 0
        p.restart_interval = self._restart_interval or 0
        p.density_unit = int(self._density.unit)
        p.density_x, p.density_y = self._density.density
        keep = []
        if self._app_segments:
            arr = (_App * len(self._app_segments))()
            for i, (nr, payload) in enumerate(self._app_segments):
                buf = (C.c_uint8 * max(1, len(payload))).from_buffer_copy(payload or b"\0")
                keep.append(buf)
                arr[i].nr, arr[i].data, arr[i].len = nr, C.cast(buf, C.POINTER(C.c_uint8)), len(payload)
            p.n_app, p.apps = len(self._app_segments), arr
            keep.append(arr)
        p._keep = keep
        return p

    def _dev(self):
        if self._device is None:
            self._device = default_device(0)
        return self._device

    def _raise(self, rc):
        raise EncodingError(rc, self._dev().last_error())

    # -- encode, :440-503 --
    def encode(self, data, width, height, color_type):
        """Returns the JFIF bytes. `data`: bytes / bytearray / numpy uint8, packed, >= w*h*bpp long."""
        dev = self._dev()
        a = _host_view(data)
        p = self._params(width, height, ColorType(color_type))
        out = C.POINTER(C.c_uint8)()
        n = C.c_size_t()
        rc = dev.lib.jpgb_encode(dev.handle, C.byref(p), a.ctypes.data if a.size else None, a.size, C.byref(out), C.byref(n))
        if rc != 0:
            self._raise(rc)
        try:
            return C.string_at(out, n.value)
        finally:
            dev.lib.jpgb_free(out)

    def encode_to(self, writer, data, width, height, color_type):
        """Encoder::new(writer, q).encode(..): bytes go to writer.write (src/writer.rs:99-106)."""
        dev = self._dev()
        a = _host_view(data)
        p = self._params(width, height, ColorType(color_type))
        err = []

        @C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(C.c_uint8), C.c_size_t)
        def cb(_user, buf, ln):
            try:
                writer.write(C.string_at(buf, ln))
                return 0
            except Exception as e:  # propagate as EncodingError::IoError
                err.append(e)
                return 1

        rc = dev.lib.jpgb_encode_to_sink(dev.handle, C.byref(p), a.ctypes.data if a.size else None, a.size,
                                         C.cast(cb, C.c_void_p), None)
        if rc != 0:
            if err:
                raise EncodingError(6, str(err[0])) from err[0]
            self._raise(rc)

    # -- encode_image<I: ImageBuffer>, :506-515 --
    def encode_image(self, image):
        """`image` mirrors the ImageBuffer trait (src/image_buffer.rs:86-98): get_jpeg_color_type() ->
        JpegColorType, width(), height(), fill_buffers(y, buffers) appending one row of samples to each
        of up to four bytearrays. The rows are gathered on the host, the planes encoded on the GPU."""
        jct = JpegColorType(image.get_jpeg_color_type())
        w, h = image.width(), image.height()
        ncomp = jct.get_num_components()
        buffers = [bytearray() for _ in range(4)]
        for y in range(h):
            image.fill_buffers(y, buffers)
        planes = [np.frombuffer(bytes(buffers[c]), dtype=np.uint8) for c in range(ncomp)]
        return self.encode_planes(planes, w, h, jct)

    def encode_planes(self, planes, width, height, jpeg_color_type):
        """Component planes (width*height samples each, taken verbatim) -> JFIF bytes."""
        dev = self._dev()
        jct = JpegColorType(jpeg_color_type)
        views = [_host_view(pl) for pl in planes]
        if len(views) != jct.get_num_components():
            raise ValueError("expected %d planes" % jct.get_num_components())
        p = self._params(width, height, ColorType(jct.as_color_type()))
        ptrs = (C.c_void_p * 4)(*([v.ctypes.data if v.size else None for v in views] + [None] * (4 - len(views))))
        out = C.POINTER(C.c_uint8)()
        n = C.c_size_t()
        rc = dev.lib.jpgb_encode_planar(dev.handle, C.byref(p), ptrs, min(v.size for v in views), C.byref(out), C.byref(n))
        if rc != 0:
            self._raise(rc)
        try:
            return C.string_at(out, n.value)
        finally:
            dev.lib.jpgb_free(out)

    def encode_batch(self, images, width, height, color_type):
        """n images of identical geometry (host memory) -> list of bytes. No reference equivalent."""
        dev = self._dev()
        views = [_host_view(im) for im in images]
        n = len(views)
        if n == 0:
            return []
        p = self._params(width, height, ColorType(color_type))
        ptrs = (C.c_void_p * n)(*[v.ctypes.data for v in views])
        outs = (C.POINTER(C.c_uint8) * n)()
        lens = (C.c_size_t * n)()
        rc = dev.lib.jpgb_encode_batch(dev.handle, C.byref(p), ptrs, min(v.size for v in views), n, outs, lens)
        if rc != 0:
            self._raise(rc)
        res = []
        for i in range(n):
            res.append(C.string_at(outs[i], lens[i]))
            dev.lib.jpgb_free(outs[i])
        return res

    def encode_batch_device(self, d_ptr, image_stride, n, width, height, color_type):
        """Device-resident batch: returns (device pointer of the files, offsets[n+1])."""
        dev = self._dev()
        p = self._params(width, height, ColorType(color_type))
        d_files = C.c_void_p()
        offs = (C.c_uint64 * (n + 1))()
        rc = dev.lib.jpgb_encode_batch_device(dev.handle, C.byref(p), C.c_void_p(d_ptr), image_stride, n, C.byref(d_files), offs)
        if rc != 0:
            self._raise(rc)
        return d_files.value, list(offs)

    def encode_batch_device_strided(self, d_ptr, n, width, height, color_type, image_stride, row_stride, plane_stride=0):
        """Device images in any row pitch, packed (plane_stride 0) or channel-planar (jpgb_device_images,
        include/jpegenc_b200.h): returns (device pointer of the files, offsets[n+1]), like encode_batch_device."""
        dev = self._dev()
        p = self._params(width, height, ColorType(color_type))
        im = _DeviceImages(d_ptr, image_stride, row_stride, plane_stride)
        d_files = C.c_void_p()
        offs = (C.c_uint64 * (n + 1))()
        rc = dev.lib.jpgb_encode_batch_device_strided(dev.handle, C.byref(p), C.byref(im), n, C.byref(d_files), offs)
        if rc != 0:
            self._raise(rc)
        return d_files.value, list(offs)

    def encode_cuda_array(self, arr, color_type, channels_first=False):
        """Encode uint8 device images where they lie: any object with `__cuda_array_interface__` (a torch CUDA tensor,
        CuPy, Numba) shaped (H, W, C) / (N, H, W, C), or (C, H, W) / (N, C, H, W) with channels_first. Crops and other
        views with a row pitch need no copy. When the interface names a stream, the encode waits for it first.
        Returns (device pointer of the files, offsets[n+1]), like encode_batch_device."""
        ct = ColorType(color_type)
        iface = arr.__cuda_array_interface__
        ptr, n, w, h, image_stride, row_stride, plane_stride = _cuda_array_layout(iface, ct.get_bytes_per_pixel(), channels_first)
        if iface.get("stream") is not None:
            self._dev().wait_stream(int(iface["stream"]))
        return self.encode_batch_device_strided(ptr, n, w, h, ct, image_stride, row_stride, plane_stride)

    # -- one large image cut into restart-aligned strips (BASELINE config 5) --
    def scan_count(self, width, height, color_type):
        p = self._params(width, height, ColorType(color_type))
        n = C.c_uint32()
        rc = load_library().jpgb_scan_count(C.byref(p), C.byref(n))
        if rc != 0:
            raise EncodingError(rc)
        return n.value

    def plan_strips(self, width, height, color_type, max_strips):
        """[(first_row, rows)] for at most max_strips strips whose boundaries are restart boundaries of
        every scan. Raises EncodingError(BadParams) if the settings do not allow strips."""
        p = self._params(width, height, ColorType(color_type))
        arr = (_Strip * max_strips)()
        n = C.c_uint32()
        rc = load_library().jpgb_plan_strips(C.byref(p), max_strips, arr, C.byref(n))
        if rc != 0:
            raise EncodingError(rc, "strips need a restart interval that divides every scan's units per MCU-row group")
        return [(arr[i].first_row, arr[i].rows) for i in range(n.value)]

    def encode_strip_device(self, d_pixels, strip_index, n_strips, first_row, rows, width, full_height, color_type, hist_total=None):
        """Encode one strip (device pointer at its first row). Returns (device pointer, piece offsets[n_scans+1]).
        With optimized Huffman tables pass the whole image's histogram (merge_strip_histograms)."""
        dev = self._dev()
        p = self._params(width, full_height, ColorType(color_type))
        st = _Strip(strip_index, n_strips, first_row, rows, full_height)
        n_scans = self.scan_count(width, full_height, color_type)
        d_bytes = C.c_void_p()
        offs = (C.c_uint64 * (n_scans + 1))()
        if hist_total is None:
            rc = dev.lib.jpgb_encode_strip_device(dev.handle, C.byref(p), C.byref(st), C.c_void_p(d_pixels), C.byref(d_bytes), offs)
        else:
            h = (C.c_uint32 * HIST_WORDS)(*[int(x) for x in hist_total])
            rc = dev.lib.jpgb_encode_strip_device_optimized(dev.handle, C.byref(p), C.byref(st), C.c_void_p(d_pixels), h, C.byref(d_bytes), offs)
        if rc != 0:
            self._raise(rc)
        return d_bytes.value, list(offs)

    def strip_histogram_device(self, d_pixels, strip_index, n_strips, first_row, rows, width, full_height, color_type):
        """Optimized tables with strips, step 1: (hist[HIST_WORDS], edge_dc[8]) of one strip (include/jpegenc_b200.h)."""
        dev = self._dev()
        p = self._params(width, full_height, ColorType(color_type))
        st = _Strip(strip_index, n_strips, first_row, rows, full_height)
        hist = (C.c_uint32 * HIST_WORDS)()
        edge = (C.c_int16 * 8)()
        rc = dev.lib.jpgb_strip_histogram_device(dev.handle, C.byref(p), C.byref(st), C.c_void_p(d_pixels), hist, edge)
        if rc != 0:
            self._raise(rc)
        return list(hist), list(edge)

    def merge_strip_histograms(self, hist_sum, edge_dc, width, full_height, color_type):
        """Step 3: hist_sum = element-wise sum of the strips' histograms, edge_dc = their edge_dc arrays in strip
        order (n_strips * 8). Returns the whole image's histogram. Host only."""
        p = self._params(width, full_height, ColorType(color_type))
        n = len(edge_dc) // 8
        hs = (C.c_uint32 * HIST_WORDS)(*[int(x) for x in hist_sum])
        ed = (C.c_int16 * (n * 8))(*[int(x) for x in edge_dc])
        out = (C.c_uint32 * HIST_WORDS)()
        rc = load_library().jpgb_merge_strip_histograms(C.byref(p), n, hs, ed, out)
        if rc != 0:
            raise EncodingError(rc)
        return list(out)

    def build_header(self, width, height, color_type):
        """SOI .. first SOS as the host planner writes them (default Huffman tables). No GPU needed."""
        p = self._params(width, height, ColorType(color_type))
        n = C.c_size_t()
        lib = load_library()
        rc = lib.jpgb_build_header(C.byref(p), None, 0, C.byref(n))
        if rc != 0:
            raise EncodingError(rc)
        buf = (C.c_uint8 * n.value)()
        lib.jpgb_build_header(C.byref(p), buf, n.value, C.byref(n))
        return bytes(buf)

    def coef_layout(self, width, height, color_type):
        p = self._params(width, height, ColorType(color_type))
        lay = _CoefLayout()
        rc = load_library().jpgb_coef_layout_for(C.byref(p), C.byref(lay))
        if rc != 0:
            raise EncodingError(rc)
        return lay

    def stage_a_device(self, d_pixels, image_stride, n, d_coef, width, height, color_type):
        """Colour + DCT + quantization only, device to device, asynchronous on the context's stream."""
        dev = self._dev()
        p = self._params(width, height, ColorType(color_type))
        rc = dev.lib.jpgb_stage_a_device(dev.handle, C.byref(p), C.c_void_p(d_pixels), image_stride, n, C.c_void_p(d_coef))
        if rc != 0:
            self._raise(rc)
