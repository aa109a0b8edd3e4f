"""ctypes binding of the CPU oracle (oracle/jpeg_oracle.c) -- TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import
this module. The product package (jpeg_encoder_b200) never does.
"""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

_DIR = os.path.dirname(os.path.abspath(__file__))

LUMA, RGB, RGBA, BGR, BGRA, YCBCR, CMYK, CMYK_AS_YCCK, YCCK = range(9)
BPP = {LUMA: 1, RGB: 3, RGBA: 4, BGR: 3, BGRA: 4, YCBCR: 3, CMYK: 4, CMYK_AS_YCCK: 4, YCCK: 4}
NCOMP = {LUMA: 1, RGB: 3, RGBA: 3, BGR: 3, BGRA: 3, YCBCR: 3, CMYK: 4, CMYK_AS_YCCK: 4, YCCK: 4}


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


_native_dir = None


def _native_path():
    """The -march=native build suits only the machine that runs it, and its users (bench.py) may run from a read-only
    tree: it goes to a temporary directory of this process, removed at exit."""
    global _native_dir
    if _native_dir is None:
        _native_dir = tempfile.mkdtemp(prefix="jpeg_oracle_native_")
        atexit.register(shutil.rmtree, _native_dir, True)
    return os.path.join(_native_dir, "liborc_native.so")


def build(native=False, force=False):
    """Compile the oracle with gcc (oracle/Makefile). Returns the path of the shared object."""
    if native:
        path = _native_path()
        if force or not os.path.exists(path):
            subprocess.check_call(["make", "-C", _DIR, "NATIVE_SO=" + path, path], stdout=subprocess.DEVNULL)
        return path
    target = "liborc.so"
    path = os.path.join(_DIR, target)
    src = os.path.join(_DIR, "jpeg_oracle.c")
    stale = (not os.path.exists(path)) or os.path.getmtime(path) < max(
        os.path.getmtime(src), os.path.getmtime(os.path.join(_DIR, "jpeg_oracle.h")))
    if force or stale:
        subprocess.check_call(["make", "-C", _DIR, target], stdout=subprocess.DEVNULL)
    return path


_libs = {}


def lib(native=False):
    if native not in _libs:
        try:
            l = C.CDLL(build(native))
        except OSError:
            l = C.CDLL(build(native, force=True))
        l.orc_encode.argtypes = [C.POINTER(_Params), C.c_void_p, C.c_size_t,
                                 C.POINTER(C.POINTER(C.c_uint8)), C.POINTER(C.c_size_t)]
        l.orc_encode.restype = C.c_int
        l.orc_free.argtypes = [C.c_void_p]
        l.orc_free.restype = None
        l.orc_coefficients.argtypes = [C.POINTER(_Params), C.c_void_p, C.c_size_t,
                                       C.POINTER(C.POINTER(C.c_int16)), C.POINTER(C.c_uint32)]
        l.orc_coefficients.restype = C.c_int
        l.orc_rgb_to_ycbcr.argtypes = [C.c_uint8, C.c_uint8, C.c_uint8, C.POINTER(C.c_uint8)]
        l.orc_fdct.argtypes = [C.POINTER(C.c_int16)]
        l.orc_fdct_i16model.argtypes = [C.POINTER(C.c_int16)]
        l.orc_fdct_simd.argtypes = [C.POINTER(C.c_int16)]
        l.orc_set_simd.argtypes = [C.c_int]
        l.orc_has_simd.restype = C.c_int
        l.orc_quant_table.argtypes = [C.c_uint8, C.POINTER(C.c_uint16), C.c_uint8, C.c_int,
                                      C.POINTER(C.c_uint16), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
        l.orc_quantize.argtypes = [C.c_int16, C.c_int32, C.c_int32]
        l.orc_quantize.restype = C.c_int16
        l.orc_get_num_bits.argtypes = [C.c_int16]
        l.orc_get_num_bits.restype = C.c_uint8
        l.orc_get_code.argtypes = [C.c_int16, C.POINTER(C.c_uint8), C.POINTER(C.c_uint16)]
        l.orc_huffman_optimized.argtypes = [C.POINTER(C.c_uint32), C.POINTER(C.c_uint8), C.POINTER(C.c_uint8)]
        l.orc_huffman_optimized.restype = C.c_int
        _libs[native] = l
    return _libs[native]


class OracleError(Exception):
    def __init__(self, code):
        super().__init__("oracle error %d" % code)
        self.code = code


def _as_bytes(data):
    if isinstance(data, np.ndarray):
        return np.ascontiguousarray(data, dtype=np.uint8).reshape(-1)
    return np.frombuffer(bytes(data), dtype=np.uint8)


def make_params(width, height, color_type, quality=90, sampling=None, qtables=(0, 0),
                progressive_scans=0, restart_interval=0, optimize_huffman=False,
                density=(0, 1, 1), app_segments=()):
    """qtables: per table either a preset index 0..8 or a sequence of 64 u16 (Custom).
    sampling: (h, v) or None for the reference default (F_2_2 below quality 90, src/encoder.rs:256-260)."""
    p = _Params()
    p.width, p.height = width, height
    p.color_type, p.quality = color_type, quality
    if sampling is None:
        sampling = (2, 2) if quality < 90 else (1, 1)
    p.sampling = (sampling[0] << 4) | sampling[1]
    for i, t in enumerate(qtables):
        if isinstance(t, int):
            p.qtable_kind[i] = t
        else:
            p.qtable_kind[i] = 9
            for k in range(64):
                p.qtable_custom[i][k] = int(t[k])
    p.progressive_scans = progressive_scans
    p.optimize_huffman = 1 if optimize_huffman else 0
    p.restart_interval = restart_interval
    p.density_unit, p.density_x, p.density_y = density
    keep = []
    if app_segments:
        arr = (_App * len(app_segments))()
        for i, (nr, payload) in enumerate(app_segments):
            buf = (C.c_uint8 * max(1, len(payload))).from_buffer_copy(bytes(payload) or b"\0")
            keep.append(buf)
            arr[i].nr, arr[i].data, arr[i].len = nr, C.cast(buf, C.POINTER(C.c_uint8)), len(payload)
        p.n_app, p.apps = len(app_segments), arr
        keep.append(arr)
    p._keep = keep
    return p


def encode(data, width, height, color_type, native=False, **kw):
    """Encoder::encode restated on the CPU (src/encoder.rs:440). Returns the JPEG bytes."""
    l = lib(native)
    p = make_params(width, height, color_type, **kw)
    a = _as_bytes(data)
    out = C.POINTER(C.c_uint8)()
    n = C.c_size_t()
    rc = l.orc_encode(C.byref(p), a.ctypes.data, a.size, C.byref(out), C.byref(n))
    if rc != 0:
        raise OracleError(rc)
    try:
        return C.string_at(out, n.value)
    finally:
        l.orc_free(out)


def coefficients(data, width, height, color_type, **kw):
    """Quantized zig-zag blocks per component over the MCU-padded grid: list of (n_blocks, 64) int16."""
    l = lib()
    p = make_params(width, height, color_type, **kw)
    a = _as_bytes(data)
    ptrs = (C.POINTER(C.c_int16) * 4)()
    counts = (C.c_uint32 * 4)()
    rc = l.orc_coefficients(C.byref(p), a.ctypes.data, a.size, ptrs, counts)
    if rc != 0:
        raise OracleError(rc)
    res = []
    for c in range(NCOMP[color_type]):
        n = counts[c]
        res.append(np.ctypeslib.as_array(ptrs[c], shape=(n, 64)).copy())
        l.orc_free(ptrs[c])
    return res


def set_simd(on, native=False):
    """CPU-baseline switch (jpeg_oracle.h): AVX2 colour + fDCT like the reference's `simd` feature."""
    lib(native).orc_set_simd(1 if on else 0)


def has_simd(native=False):
    return bool(lib(native).orc_has_simd())


def fdct(block, i16model=False, simd=False):
    a = np.ascontiguousarray(block, dtype=np.int16).reshape(64).copy()
    f = lib().orc_fdct_i16model if i16model else (lib().orc_fdct_simd if simd else lib().orc_fdct)
    f(a.ctypes.data_as(C.POINTER(C.c_int16)))
    return a


def rgb_to_ycbcr(r, g, b):
    out = (C.c_uint8 * 3)()
    lib().orc_rgb_to_ycbcr(r, g, b, out)
    return tuple(out)


def quant_table(kind, quality, luma, custom=None):
    tab = (C.c_uint16 * 64)()
    rec = (C.c_int32 * 64)()
    cor = (C.c_int32 * 64)()
    cu = (C.c_uint16 * 64)(*(custom if custom is not None else [0] * 64))
    lib().orc_quant_table(9 if custom is not None else kind, cu, quality, 1 if luma else 0, tab, rec, cor)
    return list(tab), list(rec), list(cor)


def quantize(v, recip, corr):
    return lib().orc_quantize(v, recip, corr)


def get_num_bits(v):
    return lib().orc_get_num_bits(v)


def get_code(v):
    s = C.c_uint8()
    b = C.c_uint16()
    lib().orc_get_code(v, C.byref(s), C.byref(b))
    return s.value, b.value


def huffman_optimized(freq):
    f = (C.c_uint32 * 257)(*freq)
    length = (C.c_uint8 * 16)()
    values = (C.c_uint8 * 256)()
    n = lib().orc_huffman_optimized(f, length, values)
    return list(length), list(values)[:n]
