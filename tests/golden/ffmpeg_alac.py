"""FFmpeg ALAC encoder/decoder driven through ctypes -- FIXTURE GENERATION ONLY.

Used by gen_ffmpeg_fixtures.py, and by wide_matrix.py / exotic_matrix.py when these libraries are present; never by
smoke() or bench.py's timed paths. The shared libraries are the ones the opencv-python-headless wheel bundles next to its
cv2 package; no headers come with them, so the struct offsets below were found empirically for that exact build
(libavcodec 62.11.100, SURVEY.md appendix C), and any other build is refused at import.
This is the same independent encoder + cross-decoder the reference's conformance suite uses
(tests/conformance_test.go:439-467, :518-529 of the reference).
"""
import ctypes as C
import glob
import importlib.util
import os
import struct

import numpy as np

_AVCODEC_VERSION = (62 << 16) | (11 << 8) | 100  # the build the offsets below belong to
_loaded = {}


def _libs_dir():
    spec = importlib.util.find_spec('cv2')
    if spec is None or spec.origin is None:
        raise ImportError('opencv-python-headless (the FFmpeg libraries it bundles) is not installed')
    return os.path.join(os.path.dirname(os.path.dirname(spec.origin)), 'opencv_python_headless.libs') + os.sep


_D = _libs_dir()


def _L(pat):
    path = glob.glob(_D + pat)[0]
    if path not in _loaded:
        _loaded[path] = C.CDLL(path, mode=C.RTLD_GLOBAL)
    return _loaded[path]


def _init():
    for p in ('libcrypto*', 'libssl*', 'libdrm*', 'libpng16*', 'libaom*', 'libvpx*'):
        _L(p)
    avu = _L('libavutil*')
    for p in ('libswresample*', 'libswscale*', 'libavif*'):
        _L(p)
    avc = _L('libavcodec*')
    if avc.avcodec_version() != _AVCODEC_VERSION:
        raise ImportError(f'libavcodec {avc.avcodec_version():#x}: the struct offsets here are for {_AVCODEC_VERSION:#x}')
    P = C.c_void_p
    for f, lib in (('avcodec_find_encoder_by_name', avc), ('avcodec_find_decoder_by_name', avc),
                   ('avcodec_alloc_context3', avc), ('av_packet_alloc', avc), ('av_frame_alloc', avu),
                   ('av_mallocz', avu)):
        getattr(lib, f).restype = P
    avc.avcodec_alloc_context3.argtypes = [P]
    avc.avcodec_open2.argtypes = [P, P, P]
    avu.av_mallocz.argtypes = [C.c_size_t]
    avc.avcodec_send_frame.argtypes = avc.avcodec_receive_packet.argtypes = [P, P]
    avc.avcodec_send_packet.argtypes = avc.avcodec_receive_frame.argtypes = [P, P]
    avc.av_packet_unref.argtypes = avu.av_frame_unref.argtypes = [P]
    avc.av_new_packet.argtypes = [P, C.c_int]
    avu.av_opt_set.argtypes = [P, C.c_char_p, C.c_char_p, C.c_int]
    avu.av_opt_set_int.argtypes = [P, C.c_char_p, C.c_int64, C.c_int]
    avu.av_channel_layout_from_string.argtypes = [P, C.c_char_p]
    avu.av_frame_get_buffer.argtypes = [P, C.c_int]
    return avu, avc


avu, avc = _init()
LAY = {1: b'mono', 2: b'stereo', 3: b'3.0', 4: b'4.0', 5: b'5.0', 6: b'5.1', 7: b'6.1(back)', 8: b'7.1(wide)'}
S16P, S32P = 6, 7
rd = C.string_at


def _put32(p, o, v):
    C.memmove(p + o, struct.pack('<i', v), 4)


def _ptr(p, o):
    return struct.unpack('<Q', rd(p + o, 8))[0]


def alac_encode(x, bits, sr, opts=None):
    """x: int64 [ch, n] -> (36-byte cookie, [packet bytes])."""
    ch, n = x.shape
    fmt = S16P if bits == 16 else S32P
    enc = avc.avcodec_find_encoder_by_name(b'alac')
    c = avc.avcodec_alloc_context3(enc)
    avu.av_opt_set_int(c, b'ar', sr, 0)
    avu.av_channel_layout_from_string(c + 352, LAY[ch])
    _put32(c, 348, fmt)
    if bits != 16:
        _put32(c, 652, bits)
    for k, v in (opts or {}).items():
        assert avu.av_opt_set(c, k, v, 1) == 0, (k, v)
    assert avc.avcodec_open2(c, enc, None) == 0
    cookie = rd(_ptr(c, 72), struct.unpack('<i', rd(c + 80, 4))[0])
    fr = avu.av_frame_alloc()
    pk = avc.av_packet_alloc()
    out = []

    def drain():
        while avc.avcodec_receive_packet(c, pk) == 0:
            out.append(rd(_ptr(pk, 24), struct.unpack('<i', rd(pk + 32, 4))[0]))
            avc.av_packet_unref(pk)

    for s in range(0, n, 4096):
        m = min(4096, n - s)
        _put32(fr, 112, m)
        _put32(fr, 116, fmt)
        _put32(fr, 180, sr)
        avu.av_channel_layout_from_string(fr + 384, LAY[ch])
        assert avu.av_frame_get_buffer(fr, 0) == 0
        C.memmove(fr + 136, struct.pack('<q', s), 8)
        ext = _ptr(fr, 96)
        for k in range(ch):
            b = (x[k, s:s + m].astype('<i2') if bits == 16 else (x[k, s:s + m] << (32 - bits)).astype('<i4')).tobytes()
            C.memmove(_ptr(ext, 8 * k), b, len(b))
        assert avc.avcodec_send_frame(c, fr) == 0
        avu.av_frame_unref(fr)
        drain()
    avc.avcodec_send_frame(c, None)
    drain()
    return cookie, out


def alac_decode(cookie, pkts, bits, ch, sr):
    """Independent FFmpeg decode -> int64 [ch, n]."""
    dec = avc.avcodec_find_decoder_by_name(b'alac')
    c = avc.avcodec_alloc_context3(dec)
    avu.av_opt_set_int(c, b'ar', sr, 0)
    avu.av_channel_layout_from_string(c + 352, LAY[ch])
    ed = avu.av_mallocz(len(cookie) + 64)
    C.memmove(ed, cookie, len(cookie))
    C.memmove(c + 72, struct.pack('<Q', ed), 8)
    _put32(c, 80, len(cookie))
    assert avc.avcodec_open2(c, dec, None) == 0
    fr = avu.av_frame_alloc()
    pk = avc.av_packet_alloc()
    out = [[] for _ in range(ch)]
    for pb in pkts:
        avc.av_new_packet(pk, len(pb))
        C.memmove(_ptr(pk, 24), pb, len(pb))
        rc = avc.avcodec_send_packet(c, pk)
        avc.av_packet_unref(pk)
        if rc != 0:
            raise RuntimeError(f'ffmpeg send_packet rc={rc}')
        while avc.avcodec_receive_frame(c, fr) == 0:
            m, fmt = struct.unpack('<ii', rd(fr + 112, 8))
            ext = _ptr(fr, 96)
            for k in range(ch):
                out[k].append(np.frombuffer(rd(_ptr(ext, 8 * k), m * (2 if fmt == S16P else 4)),
                                            dtype='<i2' if fmt == S16P else '<i4').astype(np.int64))
            avu.av_frame_unref(fr)
    y = np.stack([np.concatenate(o) for o in out])
    return y if bits == 16 else y >> (32 - bits)
