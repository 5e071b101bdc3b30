"""ctypes wrapper of the CPU golden model (oracle/).  TEST INFRASTRUCTURE ONLY: imported by
tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs."""
import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
LIB = os.path.join(ORACLE_DIR, "liboracle_h264.so")


class GmConfig(C.Structure):
    _fields_ = [(n, C.c_int) for n in (
        "src_width", "src_height", "src_format", "dst_width", "dst_height", "profile", "level", "qp",
        "keyframe_interval", "entropy_coding_mode", "me_range", "relax_gop", "intra4x4", "slice_rows", "sps_crop",
        "auto_level", "repeat_headers", "p_intra")]


class GmMb(C.Structure):
    _fields_ = [("type", C.c_uint8), ("i16_mode", C.c_uint8), ("chroma_mode", C.c_uint8), ("cbp", C.c_uint8),
                ("mv", C.c_int16 * 2), ("mvd", C.c_int16 * 2), ("nnz", C.c_uint8 * 27),
                ("i4_mode", C.c_uint8 * 16), ("coef", (C.c_int16 * 16) * 26)]


MB_DTYPE = np.dtype([("type", "u1"), ("i16_mode", "u1"), ("chroma_mode", "u1"), ("cbp", "u1"),
                     ("mv", "<i2", (2,)), ("mvd", "<i2", (2,)), ("nnz", "u1", (27,)), ("i4_mode", "u1", (16,)),
                     ("pad", "u1"), ("coef", "<i2", (26, 16))])

_lib = None


def build(force=False):
    src = [os.path.join(ORACLE_DIR, f) for f in ("h264_golden.c", "h264_golden.h", "h264_tables.h", "h264_decoder.c",
                                                 "h264_decoder.h")]
    if force or not os.path.exists(LIB) or any(os.path.getmtime(s) > os.path.getmtime(LIB) for s in src):
        subprocess.check_call(["make", "-s", "-C", ORACLE_DIR, "liboracle_h264.so", "golden_enc"])
    return LIB


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(LIB)
        L.gm_open.argtypes = [C.POINTER(GmConfig), C.POINTER(C.c_void_p)]
        L.gm_encode_frame.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.gm_close.argtypes = [C.c_void_p]
        for f in ("gm_coded_width", "gm_coded_height", "gm_last_frame_type"):
            getattr(L, f).argtypes = [C.c_void_p]
        L.gm_mbs.argtypes = [C.c_void_p]
        L.gm_mbs.restype = C.c_void_p
        for f in ("gm_recon", "gm_recon_unfiltered", "gm_source"):
            getattr(L, f).argtypes = [C.c_void_p, C.c_int]
            getattr(L, f).restype = C.c_void_p
        L.gm_last_sse_y.argtypes = [C.c_void_p]
        L.gm_last_sse_y.restype = C.c_double
        L.gm_write_sps.argtypes = [C.POINTER(GmConfig), C.c_void_p, C.c_int]
        L.gm_write_pps.argtypes = [C.POINTER(GmConfig), C.c_void_p, C.c_int]
        L.gm_slice_header_bits.argtypes = [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_uint32), C.POINTER(C.c_int)]
        L.gm_slice_header_bits64.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_uint64),
                                             C.POINTER(C.c_int)]
        L.gd_open.restype = C.c_void_p
        L.gd_decode.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        L.gd_error.argtypes = [C.c_void_p]
        L.gd_error.restype = C.c_char_p
        for f in ("gd_frames", "gd_width", "gd_height", "gd_crop_right", "gd_crop_bottom", "gd_close"):
            getattr(L, f).argtypes = [C.c_void_p]
        L.gd_close.restype = None
        L.gd_frame.argtypes = [C.c_void_p, C.c_int, C.c_int]
        L.gd_frame.restype = C.c_void_p
        L.gm_synth_frame.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        L.gm_cabac_code_bins.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_int, C.c_void_p, C.c_int,
                                         C.c_void_p, C.c_void_p]
        assert C.sizeof(GmMb) == MB_DTYPE.itemsize, (C.sizeof(GmMb), MB_DTYPE.itemsize)
        _lib = L
    return _lib


def align16(x):
    return (x + 15) & ~15


def make_config(width, height, qp=24, gop=25, cabac=1, fmt=0, me_range=16, profile=77, level=41, intra4x4=0,
                dst_width=None, dst_height=None, relax_gop=1, slice_rows=0, sps_crop=0, auto_level=0, repeat_headers=0, p_intra=0):
    return GmConfig(width, height, fmt, align16(width) if dst_width is None else dst_width,
                    align16(height) if dst_height is None else dst_height, profile, level, qp, gop, cabac,
                    me_range, relax_gop, intra4x4, slice_rows, sps_crop, auto_level, repeat_headers, p_intra)


def synth_frame(width, height, t, fmt=0):
    L = lib()
    y = np.empty((height, width), np.uint8)
    c = np.empty((height if fmt else height // 2, width), np.uint8)
    L.gm_synth_frame(width, height, fmt, t, y.ctypes.data, c.ctypes.data)
    return y, c


class Encoder:
    def __init__(self, cfg: GmConfig):
        self.L = lib()
        self.cfg = cfg
        self.h = C.c_void_p()
        r = self.L.gm_open(C.byref(cfg), C.byref(self.h))
        if r:
            raise OSError(-r, "gm_open failed: %d" % r)
        self.W = self.L.gm_coded_width(self.h)
        self.H = self.L.gm_coded_height(self.h)
        self.out = np.empty(self.W * self.H * 3 + 65536, np.uint8)

    def encode(self, luma, chroma) -> bytes:
        luma = np.ascontiguousarray(luma, np.uint8)
        chroma = np.ascontiguousarray(chroma, np.uint8)
        n = self.L.gm_encode_frame(self.h, luma.ctypes.data, chroma.ctypes.data, self.out.ctypes.data, self.out.size)
        if n < 0:
            raise OSError(-n, "gm_encode_frame failed: %d" % n)
        return self.out[:n].tobytes()

    def _planes(self, fn):
        out = []
        for p in range(3):
            w, h = (self.W, self.H) if p == 0 else (self.W // 2, self.H // 2)
            ptr = fn(self.h, p)
            out.append(np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_uint8)), shape=(h, w)).copy())
        return out

    def recon(self):
        return self._planes(self.L.gm_recon)

    def recon_unfiltered(self):
        return self._planes(self.L.gm_recon_unfiltered)

    def source(self):
        return self._planes(self.L.gm_source)

    def mbs(self):
        n = (self.W // 16) * (self.H // 16)
        ptr = self.L.gm_mbs(self.h)
        buf = (C.c_uint8 * (n * MB_DTYPE.itemsize)).from_address(ptr)
        return np.frombuffer(buf, dtype=MB_DTYPE).copy()

    def sse_y(self):
        return self.L.gm_last_sse_y(self.h)

    def frame_is_i(self):
        return bool(self.L.gm_last_frame_type(self.h))

    def close(self):
        if self.h:
            self.L.gm_close(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def write_sps(cfg):
    buf = np.zeros(64, np.uint8)
    n = lib().gm_write_sps(C.byref(cfg), buf.ctypes.data, 64)
    return buf[:n].tobytes()


def write_pps(cfg):
    buf = np.zeros(64, np.uint8)
    n = lib().gm_write_pps(C.byref(cfg), buf.ctypes.data, 64)
    return buf[:n].tobytes()


def slice_header_bits(frame_i, frame_p_count, cabac, first_mb=0):
    if first_mb:
        bits64, n = C.c_uint64(), C.c_int()
        lib().gm_slice_header_bits64(frame_i, frame_p_count, cabac, first_mb, C.byref(bits64), C.byref(n))
        return format(bits64.value, "0%db" % n.value)
    bits, n = C.c_uint32(), C.c_int()
    lib().gm_slice_header_bits(frame_i, frame_p_count, cabac, C.byref(bits), C.byref(n))
    return format(bits.value, "0%db" % n.value)


def cabac_code_bins(bins, frame_i, qp, hdr_bits=0, hdr_nbits=0):
    """The golden model's spec-literal CABAC coder on raw bins (uint16, the product's bin format).  Returns
    (rbsp bytes, pre-state of every bin (0 for bypass / terminate), (longest outstanding run, 1 if a carry ended it,
    slice data bits through the stop bit))."""
    bins = np.ascontiguousarray(bins, np.uint16)
    cap = 2 * bins.size + 256
    out = np.zeros(cap, np.uint8)
    pre = np.zeros(bins.size, np.uint8)
    stats = np.zeros(3, np.int32)
    n = lib().gm_cabac_code_bins(bins.ctypes.data, bins.size, frame_i, qp, hdr_bits, hdr_nbits, out.ctypes.data, cap,
                                 pre.ctypes.data, stats.ctypes.data)
    if n < 0:
        raise ValueError("gm_cabac_code_bins: %d" % n)
    return out[:n].tobytes(), pre, tuple(int(v) for v in stats)


def golden_decode(stream: bytes, crop=True):
    """The golden model's own decoder (oracle/h264_decoder.c): list of (Y, U, V) planes, like tests/avdec.decode."""
    L = lib()
    d = L.gd_open()
    buf = np.frombuffer(stream, np.uint8)
    n = L.gd_decode(d, buf.ctypes.data, buf.size)
    if n < 0:
        msg = L.gd_error(d).decode()
        L.gd_close(d)
        raise ValueError("golden decoder: " + msg)
    W, H = L.gd_width(d), L.gd_height(d)
    w, h = (W - L.gd_crop_right(d), H - L.gd_crop_bottom(d)) if crop else (W, H)
    out = []
    for i in range(n):
        planes = []
        for p, (pw, ph, cw, ch) in enumerate(((W, H, w, h), (W // 2, H // 2, w // 2, h // 2), (W // 2, H // 2, w // 2, h // 2))):
            a = np.ctypeslib.as_array(C.cast(L.gd_frame(d, i, p), C.POINTER(C.c_uint8)), shape=(ph, pw))
            planes.append(a[:ch, :cw].copy())
        out.append(tuple(planes))
    L.gd_close(d)
    return out
