"""saprobe-alac_b200 -- Python host binding over the C ABI (include/alac_b200.h).

Mirrors the reference's exported Go API name for name so the parity tests read like the reference's
own tests (/root/reference/README.md:38-54):

    ParseMagicCookie(cookie) -> PacketConfig                  config.go:47
    NewPacketDecoder(config) -> PacketDecoder                 decoder.go:90
    PacketDecoder.DecodePacket(packet) -> bytes               decoder.go:117
    PacketDecoder.DecodePackets(packets) -> (pcm list, errs)  NEW (north star): one batched GPU call
    PacketDecoder.Format() -> PCMFormat                       decoder.go:112
    NewLibraryDecoder(devices).DecodeTracks(tracks)           NEW: many tracks of mixed cookies, sharded over devices
    NewDecoder(file bytes | file object) -> Decoder           decode.go:50
    Decoder.Read(n) / Seek(ns) / Format() / Duration() / Position()   decode.go:78-190
    PacketDecoder.DecodePlanar(d_packed, d_offsets, d_sizes)  NEW: CUDA tensors in, channel-planar samples out (torch)
    LoadTrack(file bytes | file object) -> (Tensor[C, T], PCMFormat)  NEW: NewDecoder(...).ReadAll() as a CUDA tensor
    LibraryDecoder.DecodePlanar(d_packed, ..., cookies, counts)  NEW: many tracks of mixed cookies, device-resident (torch)
    LoadTracks([file bytes | file object]) -> [LoadedTrack]    NEW: LoadTrack of many files in one decode call

Errors mirror errors.go:22-34: ErrConfig, ErrNoTrack, ErrDecode (exception classes; `.status` is the
status word of the C ABI, `str()` the reference's wrapped message).

All decoding happens in libalacb200.so (hand-written CUDA, no CPU fallback): importing this module
fails loudly if the library is missing, and creating a decoder fails if no CUDA device is usable.
The directory name contains a hyphen, so load it with `load_package()` from the repo-root helper
`alac_b200_loader.py` (registered in sys.modules as `saprobe_alac_b200`).
"""
import ctypes as C
import os
from dataclasses import dataclass

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# ALACB200_LIB: developer override (an experiment or `make dev` build of the same ABI, e.g. libalacb200_dev.so)
LIB_PATH = os.environ.get('ALACB200_LIB') or os.path.join(_HERE, 'libalacb200.so')

# ---- API results / status words (include/alac_b200.h) ----------------------------------------------
OK = 0
E_ARG, E_CUDA, E_NO_DEVICE, E_NOMEM, E_CONFIG, E_IO, E_NO_TRACK = -1, -2, -3, -4, -5, -6, -7
ST_OK = 0
ST_INVALID_COOKIE, ST_UNSUPPORTED_VERSION, ST_UNSUPPORTED_ELEMENT, ST_INVALID_HEADER = 1, 2, 3, 4
ST_INVALID_SHIFT, ST_BITSTREAM_OVERRUN, ST_SAMPLE_OVERRUN, ST_BIT_DEPTH = 5, 6, 7, 8
ST_REF_PANIC, ST_UNSUPPORTED_CONFIG, ST_IO_TRUNCATED = 9, 10, 11
SAMPLES_S16, SAMPLES_S32, SAMPLES_F32 = 1, 2, 3


class PacketConfig(C.Structure):
    """PacketConfig, config.go:27-38 == alacb200_config."""
    _fields_ = [('FrameLength', C.c_uint32), ('BitDepth', C.c_uint8), ('NumChannels', C.c_uint8),
                ('PB', C.c_uint8), ('MB', C.c_uint8), ('KB', C.c_uint8), ('_reserved', C.c_uint8),
                ('MaxRun', C.c_uint16), ('MaxFrameBytes', C.c_uint32), ('AvgBitRate', C.c_uint32),
                ('SampleRate', C.c_uint32)]

    def __repr__(self):
        return ('PacketConfig(' + ', '.join(f'{n}={getattr(self, n)}' for n, _ in self._fields_ if n[0] != '_') + ')')


@dataclass(frozen=True)
class PCMFormat:
    """PCMFormat, format.go:20-24."""
    SampleRate: int
    BitDepth: int
    Channels: int


class _PcmFormatC(C.Structure):
    _fields_ = [('sample_rate', C.c_int32), ('bit_depth', C.c_int32), ('channels', C.c_int32)]


class Profile(C.Structure):
    _fields_ = [('launches_decode', C.c_uint64), ('ms_decode', C.c_double)]


class TrackDesc(C.Structure):
    """alacb200_track_desc (include/alac_b200.h): one track of a library batch."""
    _fields_ = [('cookie', C.c_void_p), ('cookie_len', C.c_size_t), ('data', C.c_void_p), ('data_len', C.c_uint64),
                ('offsets', C.c_void_p), ('sizes', C.c_void_p), ('n', C.c_uint32), ('reserved', C.c_uint32),
                ('pcm_out', C.c_void_p), ('out_stride', C.c_uint64), ('out_bytes', C.c_void_p), ('status', C.c_void_p),
                ('config', PacketConfig), ('track_status', C.c_int32), ('result', C.c_int32), ('device', C.c_int32),
                ('reserved2', C.c_int32)]


class PlanarTrackDesc(C.Structure):
    """alacb200_planar_track (include/alac_b200.h): one track of a multi-track planar call."""
    _fields_ = [('cookie', C.c_void_p), ('cookie_len', C.c_size_t), ('n', C.c_uint32), ('reserved', C.c_uint32),
                ('d_out', C.c_void_p), ('channel_stride', C.c_uint64), ('config', PacketConfig), ('track_status', C.c_int32),
                ('result', C.c_int32)]


class SampleInfo(C.Structure):
    """SampleInfo, internal/mp4/mp4.go:28-31."""
    _fields_ = [('Offset', C.c_uint64), ('Size', C.c_uint32), ('_reserved', C.c_uint32)]


# ---- errors (errors.go:22-34) -------------------------------------------------------------------------
class AlacError(Exception):
    status = 0


class ErrConfig(AlacError):
    """invalid configuration"""


class ErrNoTrack(AlacError):
    """no track found"""


class ErrDecode(AlacError):
    """decode failed"""


class CudaError(RuntimeError):
    """The CUDA path is unusable (no device, driver failure). There is no CPU fallback."""


_CONFIG_CODES = (ST_INVALID_COOKIE, ST_UNSUPPORTED_VERSION, ST_BIT_DEPTH, ST_UNSUPPORTED_CONFIG)


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(f'{LIB_PATH} is missing: build it with `python -c "import __graft_entry__ as g; g.build()"` '
                          '(nvcc, sm_100a). saprobe-alac_b200 has no CPU fallback.')
    L = C.CDLL(LIB_PATH)
    vp, u8p = C.c_void_p, C.c_char_p
    sig = {
        'alacb200_parse_cookie': (C.c_int32, [u8p, C.c_size_t, C.POINTER(PacketConfig)]),
        'alacb200_bytes_per_sample': (C.c_int32, [C.c_uint8]),
        'alacb200_create': (C.c_int32, [C.POINTER(PacketConfig), C.c_int, C.POINTER(vp), C.POINTER(C.c_int32)]),
        'alacb200_destroy': (None, [vp]),
        'alacb200_format': (C.c_int32, [vp, C.POINTER(_PcmFormatC)]),
        'alacb200_get_config': (C.c_int32, [vp, C.POINTER(PacketConfig)]),
        'alacb200_max_packet_pcm_bytes': (C.c_uint64, [vp]),
        'alacb200_decode_packets': (C.c_int32, [vp, vp, C.c_uint64, vp, vp, C.c_uint32, vp, C.c_uint64, vp, vp]),
        'alacb200_arena': (C.c_int32, [vp, C.c_uint64, C.c_uint64, C.POINTER(vp), C.POINTER(vp)]),
        'alacb200_library_create': (C.c_int32, [C.POINTER(C.c_int), C.c_int, C.POINTER(vp)]),
        'alacb200_library_destroy': (None, [vp]),
        'alacb200_library_devices': (C.c_int32, [vp]),
        'alacb200_library_decode_tracks': (C.c_int32, [vp, C.POINTER(TrackDesc), C.c_uint32]),
        'alacb200_decode_packets_device': (C.c_int32, [vp, vp, C.c_uint64, vp, vp, C.c_uint32, vp, C.c_uint64, vp, vp, vp]),
        'alacb200_decode_planar_device': (C.c_int32, [vp, vp, C.c_uint64, vp, vp, C.c_uint32, C.c_int32, vp, C.c_uint64, vp, vp, vp]),
        'alacb200_library_decode_planar_device': (C.c_int32, [vp, C.c_int, vp, C.c_uint64, vp, vp, C.POINTER(PlanarTrackDesc),
                                                              C.c_uint32, C.c_int32, vp, vp, vp]),
        'alacb200_pinned_alloc': (vp, [C.c_size_t]),
        'alacb200_pinned_free': (None, [vp]),
        'alacb200_strerror': (C.c_char_p, [C.c_int32]),
        'alacb200_format_error': (C.c_size_t, [C.c_int32, C.c_char_p, C.c_size_t]),
        'alacb200_last_error': (C.c_char_p, []),
        'alacb200_device_count': (C.c_int32, []),
        'alacb200_set_profiling': (C.c_int32, [vp, C.c_int]),
        'alacb200_get_profile': (C.c_int32, [vp, C.POINTER(Profile)]),
        'alacb200_mp4_find_alac_track': (C.c_int32, [vp, C.c_uint64, C.POINTER(vp)]),
        'alacb200_mp4_free_track': (None, [vp]),
        'alacb200_mp4_cookie': (vp, [vp, C.POINTER(C.c_size_t)]),
        'alacb200_mp4_samples': (C.POINTER(SampleInfo), [vp, C.POINTER(C.c_uint64)]),
        'alacb200_mp4_error': (C.c_char_p, [vp]),
    }
    for name, (res, args) in sig.items():
        f = getattr(L, name)
        f.restype, f.argtypes = res, args
    return L


lib = _load()
ABI_SYMBOLS = ('alacb200_parse_cookie alacb200_bytes_per_sample alacb200_create alacb200_destroy alacb200_format '
               'alacb200_get_config alacb200_max_packet_pcm_bytes alacb200_decode_packets alacb200_arena '
               'alacb200_library_create alacb200_library_destroy alacb200_library_devices '
               'alacb200_library_decode_tracks alacb200_decode_packets_device alacb200_decode_planar_device '
               'alacb200_library_decode_planar_device alacb200_pinned_alloc alacb200_pinned_free alacb200_strerror '
               'alacb200_format_error alacb200_last_error alacb200_device_count alacb200_set_profiling '
               'alacb200_get_profile alacb200_mp4_find_alac_track alacb200_mp4_free_track alacb200_mp4_cookie '
               'alacb200_mp4_samples alacb200_mp4_error').split()


def format_error(status: int) -> str:
    buf = C.create_string_buffer(256)
    lib.alacb200_format_error(int(status), buf, 256)
    return buf.value.decode()


def error_from_status(status: int, prefix: str = '') -> AlacError:
    """Rebuild the reference's error chain from a status word (what the cgo shim does in Go)."""
    cls = ErrConfig if (int(status) & 0xff) in _CONFIG_CODES else ErrDecode
    err = cls(prefix + format_error(status))
    err.status = int(status)
    return err


def _check(rc: int, what: str):
    if rc != OK:
        raise CudaError(f'{what} failed (rc={rc}): {lib.alacb200_last_error().decode()}')


def _config_status(config: PacketConfig) -> int:
    """NewPacketDecoder's checks of a parsed cookie (decoder.go:90-110): ST_OK or the status it fails with."""
    if lib.alacb200_bytes_per_sample(config.BitDepth) == 0:
        return ST_BIT_DEPTH
    if not (1 <= config.NumChannels <= 8 and 1 <= config.FrameLength <= 65536):
        return ST_UNSUPPORTED_CONFIG
    return ST_OK


def _config_error(status: int, config: PacketConfig) -> AlacError:
    """The error NewPacketDecoder raises for a cookie that fails its checks with `status`."""
    err = error_from_status(status)
    if status == ST_BIT_DEPTH:
        err.args = (f'{err.args[0]}: {config.BitDepth}',)  # decoder.go:92
    return err


def _planar_type(torch, dtype, bit_depths=()):
    """dtype (None: float32) -> (torch dtype, SAMPLES_*), or ValueError for a dtype the planar path does not produce or
    int16 for a stream that is not 16-bit."""
    dtype = torch.float32 if dtype is None else dtype
    types = {torch.int16: SAMPLES_S16, torch.int32: SAMPLES_S32, torch.float32: SAMPLES_F32}
    if dtype not in types:
        raise ValueError(f'DecodePlanar: dtype must be torch.int16, torch.int32 or torch.float32, not {dtype}')
    for bits in bit_depths:
        if dtype == torch.int16 and bits != 16:
            raise ValueError(f'DecodePlanar: torch.int16 holds 16-bit streams only, this one is {bits}-bit')
    return dtype, types[dtype]


def _check_device_tensors(who, dev, **tensors):
    import torch
    want = {'d_packed': torch.uint8, 'd_offsets': torch.int64, 'd_sizes': torch.int32}
    for name, t in tensors.items():
        if t.device != dev or t.dtype != want[name] or not t.is_contiguous():
            raise ValueError(f'{who}: {name} must be a contiguous {want[name]} tensor on {dev}')


# ---- config.go ----------------------------------------------------------------------------------------
def ParseMagicCookie(cookie: bytes) -> PacketConfig:
    cfg = PacketConfig()
    cookie = bytes(cookie) if cookie is not None else b''
    st = lib.alacb200_parse_cookie(cookie, len(cookie), C.byref(cfg))
    if st != ST_OK:
        raise error_from_status(st)
    return cfg


def BytesPerSample(depth: int) -> int:
    n = lib.alacb200_bytes_per_sample(depth)
    if n == 0:
        raise ValueError(f'alac: BytesPerSample called with unsupported bit depth {depth}')  # format.go:32 panics
    return n


def pack_packets(packets, align=16):
    """Host packer: list of packet bytes -> (packed u8 [+64 B pad], offsets u64, sizes u32), 16-byte aligned."""
    sizes = np.fromiter((len(p) for p in packets), dtype=np.uint32, count=len(packets))
    padded = (sizes.astype(np.uint64) + (align - 1)) // align * align
    offsets = np.zeros(len(packets), dtype=np.uint64)
    if len(packets) > 1:
        offsets[1:] = np.cumsum(padded)[:-1]
    total = int(padded.sum()) if len(packets) else 0
    packed = np.zeros(total + 64, dtype=np.uint8)
    for p, o in zip(packets, offsets):
        packed[int(o):int(o) + len(p)] = np.frombuffer(p, dtype=np.uint8)
    return packed, offsets, sizes


def shard_ranges(weights, world: int):
    """Contiguous [lo, hi) ranges, one per rank, balanced by `weights` (compressed bytes per packet or per
    track). Packets/tracks are independent (decoder.go:79-87), so multi-GPU decode is a plain partition:
    no collective on the data path, output order = input order (SURVEY.md section 8e)."""
    w = np.asarray(weights, dtype=np.float64)
    n = len(w)
    world = max(1, int(world))
    if n == 0:
        return [(0, 0)] * world
    cum = np.concatenate([[0.0], np.cumsum(w)])
    total = cum[-1]
    bounds = [0]
    for r in range(1, world):
        target = total * r / world
        k = int(np.searchsorted(cum, target, side='left'))
        k = max(bounds[-1], min(k, n))
        bounds.append(k)
    bounds.append(n)
    return [(bounds[r], bounds[r + 1]) for r in range(world)]


# ---- decoder.go ---------------------------------------------------------------------------------------
class PacketDecoder:
    """PacketDecoder, decoder.go:79-128, on one CUDA device."""

    def __init__(self, config: PacketConfig, device: int = 0):
        self._h = C.c_void_p()
        st = C.c_int32(0)
        rc = lib.alacb200_create(C.byref(config), device, C.byref(self._h), C.byref(st))
        if rc == E_CONFIG:
            raise _config_error(st.value, config)
        _check(rc, 'alacb200_create')
        self.config = config
        self.device = device
        self.frame_bytes = int(lib.alacb200_max_packet_pcm_bytes(self._h))

    def close(self):
        if getattr(self, '_h', None):
            lib.alacb200_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # interpreter shutdown: the module globals may already be gone
            pass

    def Format(self) -> PCMFormat:
        f = _PcmFormatC()
        _check(lib.alacb200_format(self._h, C.byref(f)), 'alacb200_format')
        return PCMFormat(f.sample_rate, f.bit_depth, f.channels)

    # -- batched entry points ------------------------------------------------------------------------
    def decode_packed(self, packed, offsets, sizes, out=None, out_stride=None):
        """Raw batched call on host arrays -> (pcm [n, out_stride] u8, out_bytes u32 [n], status i32 [n]). `packed` may be
        any byte buffer the packets live in (a packed array or a whole file image)."""
        n = len(sizes)
        out_stride = out_stride or (self.frame_bytes + 3) // 4 * 4
        if out is None:
            out = np.zeros((n, out_stride), dtype=np.uint8)
        nb = np.zeros(n, dtype=np.uint32)
        st = np.zeros(n, dtype=np.int32)
        packed = np.ascontiguousarray(packed, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        sizes = np.ascontiguousarray(sizes, dtype=np.uint32)
        rc = lib.alacb200_decode_packets(self._h, packed.ctypes.data, packed.nbytes, offsets.ctypes.data, sizes.ctypes.data, n,
                                         out.ctypes.data, out_stride, nb.ctypes.data, st.ctypes.data)
        _check(rc, 'alacb200_decode_packets')
        return out, nb, st

    def _arena(self, in_bytes, out_bytes):
        """The decoder's own pinned staging (grow-only): -> (in u8 [in_bytes], out u8 [out_bytes]) views."""
        pi, po = C.c_void_p(), C.c_void_p()
        _check(lib.alacb200_arena(self._h, in_bytes, out_bytes, C.byref(pi), C.byref(po)), 'alacb200_arena')
        a = np.ctypeslib.as_array(C.cast(pi, C.POINTER(C.c_uint8)), shape=(max(in_bytes, 1),))
        b = np.ctypeslib.as_array(C.cast(po, C.POINTER(C.c_uint8)), shape=(max(out_bytes, 1),))
        return a, b

    def decode_in_place(self, data_ptr, data_len, offsets, sizes):
        """Packets read in place from `data_ptr` (a pinned file image or packed buffer) -> (pcm rows, out_bytes, status);
        the PCM lands in the decoder's pinned arena (valid until the next call)."""
        n = len(sizes)
        stride = (self.frame_bytes + 3) // 4 * 4
        _, out = self._arena(0, n * stride)
        out = out[:n * stride].reshape(n, stride)
        nb = np.zeros(n, dtype=np.uint32)
        st = np.zeros(n, dtype=np.int32)
        rc = lib.alacb200_decode_packets(self._h, data_ptr, data_len, offsets.ctypes.data, sizes.ctypes.data, n,
                                         out.ctypes.data, stride, nb.ctypes.data, st.ctypes.data)
        _check(rc, 'alacb200_decode_packets')
        return out, nb, st

    def DecodePackets(self, packets):
        """Batched DecodePacket: -> (list of PCM bytes or None, list of error or None). The packets are packed into the
        decoder's pinned arena and the PCM comes back through it: no allocation of pinned memory per call."""
        n = len(packets)
        if n == 0:
            return [], []
        sizes = np.fromiter((len(p) for p in packets), dtype=np.uint32, count=n)
        padded = (sizes.astype(np.uint64) + 15) // 16 * 16
        offsets = np.zeros(n, dtype=np.uint64)
        if n > 1:
            offsets[1:] = np.cumsum(padded)[:-1]
        total = int(padded.sum())
        stride = (self.frame_bytes + 3) // 4 * 4
        a_in, a_out = self._arena(total, n * stride)
        for p, o in zip(packets, offsets):
            a_in[int(o):int(o) + len(p)] = np.frombuffer(p, dtype=np.uint8)
        out = a_out[:n * stride].reshape(n, stride)
        nb = np.zeros(n, dtype=np.uint32)
        st = np.zeros(n, dtype=np.int32)
        rc = lib.alacb200_decode_packets(self._h, a_in.ctypes.data, total, offsets.ctypes.data, sizes.ctypes.data, n,
                                         out.ctypes.data, stride, nb.ctypes.data, st.ctypes.data)
        _check(rc, 'alacb200_decode_packets')
        pcm, errs = [], []
        for i in range(n):
            if st[i] == ST_OK:
                pcm.append(out[i, :nb[i]].tobytes())  # a fresh buffer per packet, like decoder.go:120
                errs.append(None)
            else:
                pcm.append(None)
                errs.append(error_from_status(int(st[i])))
        return pcm, errs

    def DecodePacket(self, packet: bytes) -> bytes:
        pcm, errs = self.DecodePackets([bytes(packet)])
        if errs[0] is not None:
            raise errs[0]
        return pcm[0]

    def DecodePlanar(self, d_packed, d_offsets, d_sizes, dtype=None):
        """Device-resident batch -> channel-planar samples, enqueued on torch.cuda.current_stream() without a host
        synchronisation. d_packed: uint8 CUDA tensor the packets live in (16-byte aligned, padded to a multiple of 16
        bytes, every packet inside it); d_offsets: int64 [n]; d_sizes: int32 [n]; all on this decoder's device.
        dtype: torch.float32 (default; full scale is [-1, 1)), torch.int32, or torch.int16 (16-bit streams only).
        -> (samples [channels, n * frame_length], frame_start int64 [n + 1], status int32 [n]): packet i's frames are
        samples[:, frame_start[i]:frame_start[i + 1]], a failed packet has none, frame_start[n] is the total, and
        samples past the total are not written."""
        import torch
        dtype, sample_type = _planar_type(torch, dtype, (self.config.BitDepth,))
        dev = torch.device('cuda', self.device)
        _check_device_tensors('DecodePlanar', dev, d_packed=d_packed, d_offsets=d_offsets, d_sizes=d_sizes)
        n = d_sizes.numel()
        if d_offsets.numel() != n:
            raise ValueError('DecodePlanar: d_offsets and d_sizes differ in length')
        with torch.cuda.device(dev):
            samples = torch.empty((self.config.NumChannels, n * self.config.FrameLength), dtype=dtype, device=dev)
            frame_start = torch.empty(n + 1, dtype=torch.int64, device=dev)
            status = torch.empty(n, dtype=torch.int32, device=dev)
            rc = lib.alacb200_decode_planar_device(self._h, d_packed.data_ptr(), d_packed.numel(), d_offsets.data_ptr(),
                                                   d_sizes.data_ptr(), n, sample_type, samples.data_ptr(), samples.shape[1],
                                                   frame_start.data_ptr(), status.data_ptr(), torch.cuda.current_stream(dev).cuda_stream)
        _check(rc, 'alacb200_decode_planar_device')
        return samples, frame_start, status

    # -- profiling -----------------------------------------------------------------------------------
    def set_profiling(self, on: bool):
        _check(lib.alacb200_set_profiling(self._h, int(on)), 'alacb200_set_profiling')

    def get_profile(self) -> Profile:
        p = Profile()
        _check(lib.alacb200_get_profile(self._h, C.byref(p)), 'alacb200_get_profile')
        return p


def NewPacketDecoder(config: PacketConfig, device: int = 0) -> PacketDecoder:
    return PacketDecoder(config, device)


# ---- library batches: many tracks, mixed cookies, several devices ------------------------------------
@dataclass
class Track:
    """One track of a library batch: its cookie and the bytes + sample table its packets live in (a packed buffer from
    pack_packets, or a whole M4A image with FindALACTrack's table -- read in place, never re-packed)."""
    cookie: bytes
    data: np.ndarray     # uint8
    offsets: np.ndarray  # uint64 [n]
    sizes: np.ndarray    # uint32 [n]


@dataclass
class TrackResult:
    config: PacketConfig = None
    err: Exception = None        # ErrConfig for a bad cookie / unsupported depth: the track has no decoder
    pcm: np.ndarray = None       # uint8 [n, stride]; packet i is pcm[i, :out_bytes[i]]
    out_bytes: np.ndarray = None
    status: np.ndarray = None    # status word per packet (error_from_status rebuilds the reference's error)
    device: int = -1

    def packet(self, i) -> bytes:
        if self.status[i] != ST_OK:
            raise error_from_status(int(self.status[i]))
        return self.pcm[i, :self.out_bytes[i]].tobytes()

    def pcm_bytes(self) -> bytes:
        return b''.join(self.packet(i) for i in range(len(self.status)))


class LibraryDecoder:
    """Decodes whole libraries: any mix of cookies (a PacketDecoder holds one, decoder.go:79-87), contiguous track ranges
    per device balanced by compressed bytes, one submitting host thread per device, no collective (SURVEY.md 8e)."""

    def __init__(self, devices=(0,)):
        devs = (C.c_int * len(devices))(*devices)
        self._h = C.c_void_p()
        _check(lib.alacb200_library_create(devs, len(devices), C.byref(self._h)), 'alacb200_library_create')
        self.devices = tuple(devices)

    def close(self):
        if getattr(self, '_h', None):
            lib.alacb200_library_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def DecodeTracks(self, tracks, out=None):
        """tracks: [Track] -> [TrackResult]. `out`: optional list of preallocated uint8 [n, stride] arrays (e.g. pinned)."""
        nt = len(tracks)
        descs = (TrackDesc * max(nt, 1))()
        keep, results = [], []
        for t, tr in enumerate(tracks):
            d = descs[t]
            cookie = np.frombuffer(bytes(tr.cookie) if tr.cookie is not None else b'', dtype=np.uint8)
            data = np.ascontiguousarray(tr.data, dtype=np.uint8)
            offs = np.ascontiguousarray(tr.offsets, dtype=np.uint64)
            sizes = np.ascontiguousarray(tr.sizes, dtype=np.uint32)
            n = len(sizes)
            cfg = PacketConfig()
            st = lib.alacb200_parse_cookie(bytes(tr.cookie) if tr.cookie is not None else b'', len(cookie), C.byref(cfg))
            bps = lib.alacb200_bytes_per_sample(cfg.BitDepth) if st == ST_OK else 0
            stride = (cfg.FrameLength * cfg.NumChannels * bps + 3) // 4 * 4 if bps else 4
            ok_shape = st == ST_OK and _config_status(cfg) == ST_OK
            pcm = out[t] if out is not None else (np.zeros((n, stride), dtype=np.uint8) if ok_shape else np.zeros((0, 4), dtype=np.uint8))
            nb = np.zeros(n, dtype=np.uint32)
            stt = np.zeros(n, dtype=np.int32)
            d.cookie, d.cookie_len = cookie.ctypes.data if len(cookie) else None, len(cookie)
            d.data, d.data_len = data.ctypes.data, data.nbytes
            d.offsets, d.sizes, d.n = offs.ctypes.data, sizes.ctypes.data, n
            d.pcm_out, d.out_stride = pcm.ctypes.data, (pcm.shape[1] if pcm.ndim == 2 and pcm.shape[0] else stride)
            d.out_bytes, d.status = nb.ctypes.data, stt.ctypes.data
            keep.append((cookie, data, offs, sizes))
            results.append(TrackResult(pcm=pcm, out_bytes=nb, status=stt))
        rc = lib.alacb200_library_decode_tracks(self._h, descs, nt)
        _check(rc, 'alacb200_library_decode_tracks')
        for t, r in enumerate(results):
            d = descs[t]
            r.config = PacketConfig.from_buffer_copy(d.config)
            r.device = d.device
            if d.result == E_CONFIG:
                r.err = _config_error(d.track_status, r.config)
            elif d.result != OK:
                r.err = CudaError(f'track {t}: rc={d.result}')
        del keep
        return results

    def DecodePlanar(self, d_packed, d_offsets, d_sizes, cookies, counts, dtype=None, device=None):
        """Device-resident packets of many tracks -> channel-planar samples per track, enqueued on
        torch.cuda.current_stream() without a host synchronisation: the multi-track PacketDecoder.DecodePlanar.

        The packet table is shared: d_offsets int64 [N] (absolute in d_packed), d_sizes int32 [N], track t owning the
        next counts[t] rows, track 0 first; d_packed as for PacketDecoder.DecodePlanar; all on cuda:device (default: the
        library's first device, which must be one of its devices). cookies[t] is track t's magic cookie. Adjacent
        tracks of one kernel config share their launches, so a table ordered by config is one decode launch per config.
        -> (samples, frame_start int64 [N + T], status int32 [N], errors):
          samples[t]   [channels_t, counts[t] * frame_length_t] of dtype, or None for a track whose cookie fails
                       ParseMagicCookie + NewPacketDecoder (its error is errors[t], as LibraryDecoder.DecodeTracks
                       reports it; its rows get that status word). All tracks' samples are views of one allocation.
          frame_start  track t's counts[t] + 1 entries start at (its first row + t): its packet i's frames are
                       samples[t][:, fs[i]:fs[i + 1]], a failed packet has none, fs[counts[t]] is its total, and
                       samples past the total are not written."""
        import torch
        device = self.devices[0] if device is None else device
        dtype, sample_type = _planar_type(torch, dtype)
        dev = torch.device('cuda', device)
        _check_device_tensors('LibraryDecoder.DecodePlanar', dev, d_packed=d_packed, d_offsets=d_offsets, d_sizes=d_sizes)
        counts = [int(c) for c in counts]
        nt, rows = len(cookies), sum(counts)
        if len(counts) != nt or d_offsets.numel() != rows or d_sizes.numel() != rows:
            raise ValueError('LibraryDecoder.DecodePlanar: one count per cookie, and sum(counts) rows in d_offsets and d_sizes')
        descs = (PlanarTrackDesc * max(nt, 1))()
        cookies = [np.frombuffer(bytes(c) if c is not None else b'', dtype=np.uint8) for c in cookies]
        esz = torch.empty((), dtype=dtype).element_size()
        spans, total = [], 0  # per track: (first element, channels, channel stride) of its samples in one allocation
        for t in range(nt):
            cfg = PacketConfig()
            ok = lib.alacb200_parse_cookie(cookies[t].tobytes(), len(cookies[t]), C.byref(cfg)) == ST_OK and _config_status(cfg) == ST_OK
            stride = counts[t] * cfg.FrameLength if ok else 0
            spans.append((total, cfg.NumChannels if ok else 0, stride))
            total += -(-cfg.NumChannels * stride * esz // 16) * 16 // esz if ok else 0  # every track starts 16-byte aligned
        with torch.cuda.device(dev):
            flat = torch.empty(max(total, 1), dtype=dtype, device=dev)
            frame_start = torch.empty(rows + nt, dtype=torch.int64, device=dev)
            status = torch.empty(rows, dtype=torch.int32, device=dev)
            for t in range(nt):
                d = descs[t]
                d.cookie, d.cookie_len = cookies[t].ctypes.data if len(cookies[t]) else None, len(cookies[t])
                d.n, d.channel_stride = counts[t], spans[t][2]
                d.d_out = flat.data_ptr() + spans[t][0] * esz
            rc = lib.alacb200_library_decode_planar_device(self._h, device, d_packed.data_ptr(), d_packed.numel(), d_offsets.data_ptr(),
                                                           d_sizes.data_ptr(), descs, nt, sample_type, frame_start.data_ptr(),
                                                           status.data_ptr(), torch.cuda.current_stream(dev).cuda_stream)
        if rc == E_ARG:
            raise ValueError(f'LibraryDecoder.DecodePlanar: {lib.alacb200_last_error().decode()}')
        _check(rc, 'alacb200_library_decode_planar_device')
        samples, errors = [], []
        for t in range(nt):
            d = descs[t]
            if d.result == E_CONFIG:
                samples.append(None)
                errors.append(_config_error(d.track_status, PacketConfig.from_buffer_copy(d.config)))
            else:
                a, ch, stride = spans[t]
                samples.append(flat[a:a + ch * stride].view(ch, stride))
                errors.append(None)
        return samples, frame_start, status, errors


def NewLibraryDecoder(devices=(0,)) -> LibraryDecoder:
    return LibraryDecoder(devices)


# ---- internal/mp4 ------------------------------------------------------------------------------------
def FindALACTrack(data: bytes):
    """FindALACTrack, internal/mp4/mp4.go:233-300 -> (cookie bytes, [(offset, size)])."""
    data = bytes(data)
    t = C.c_void_p()
    rc = lib.alacb200_mp4_find_alac_track(data, len(data), C.byref(t))
    try:
        if rc != OK:
            e = ErrNoTrack('no track found: ' + lib.alacb200_mp4_error(t).decode())  # decode.go:53
            raise e
        n = C.c_size_t()
        p = lib.alacb200_mp4_cookie(t, C.byref(n))
        cookie = C.string_at(p, n.value) if p else b''
        cnt = C.c_uint64()
        sp = lib.alacb200_mp4_samples(t, C.byref(cnt))
        samples = [(sp[i].Offset, sp[i].Size) for i in range(cnt.value)]
        return cookie, samples
    finally:
        lib.alacb200_mp4_free_track(t)


# ---- decode.go ----------------------------------------------------------------------------------------
_NS = 1_000_000_000


def _open_track(rs):
    """NewDecoder's container steps (decode.go:50-60): -> (file bytes, PacketConfig, [(offset, size)], cookie)."""
    data = rs if isinstance(rs, (bytes, bytearray, memoryview)) else rs.read()
    data = bytes(data)
    cookie, samples = FindALACTrack(data)
    try:
        config = ParseMagicCookie(cookie)
    except AlacError as e:
        e.args = ('parsing ALAC config: ' + e.args[0],)  # decode.go:58
        raise
    return data, config, samples, cookie


def _packet_error(idx: int, status: int) -> AlacError:
    """The error Read returns for packet idx that failed with `status` (decode.go:181)."""
    item = error_from_status(status)
    err = type(item)(f'decoding packet {idx}: {item.args[0]}')
    err.status = item.status
    return err


class Decoder:
    """Streaming Decoder, decode.go:32-190, with a GPU read-ahead window behind Read/Seek.

    The reference decodes one packet per Read loop iteration (decode.go:159-186); here Read pulls a
    window of `window` packets through one batched GPU call and serves bytes from it. Packet order,
    io.Reader semantics (short reads, EOF as b''), Seek's packet alignment and Duration's over-count
    of a partial last packet (decode.go:82-88) are unchanged.
    """

    def __init__(self, rs, device: int = 0, window: int = 2048):
        data, config, samples, _ = _open_track(rs)
        self.dec = NewPacketDecoder(config, device)
        # the file image lives in pinned memory for the life of the decoder: every window is read in place from it
        # (image + sample-table offsets straight to the C ABI, asynchronous H2D), nothing is re-packed
        self._img_len = len(data)
        self._img_ptr = lib.alacb200_pinned_alloc(max(1, self._img_len))
        if not self._img_ptr:
            raise CudaError('alacb200_pinned_alloc failed: ' + lib.alacb200_last_error().decode())
        C.memmove(self._img_ptr, data, self._img_len)
        self.samples = samples
        self._offs = np.array([o for o, _ in samples], dtype=np.uint64)
        self._sizes = np.array([z for _, z in samples], dtype=np.uint32)
        self.sampleIdx = 0
        self._window = max(1, int(window))
        self._ready = None    # (pcm rows, out_bytes, status) of packets [self._ready_base, ...)
        self._ready_n = 0
        self._ready_base = 0
        self._buf = b''
        self._bufOff = 0
        self._eof = False

    def close(self):
        if getattr(self, '_img_ptr', None):
            self.dec.close()
            lib.alacb200_pinned_free(self._img_ptr)
            self._img_ptr = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def Format(self) -> PCMFormat:
        return self.dec.Format()

    def Duration(self) -> int:
        """nanoseconds, decode.go:82-88"""
        c = self.dec.config
        return len(self.samples) * c.FrameLength * _NS // c.SampleRate

    def Position(self) -> int:
        c = self.dec.config
        return self.sampleIdx * c.FrameLength * _NS // c.SampleRate

    def Seek(self, t_ns: int) -> int:
        """decode.go:103-124: packet-granular, clamped to [0, len(samples)]; returns the aligned time."""
        c = self.dec.config
        target_frame = int((t_ns / _NS) * float(c.SampleRate))
        q = abs(target_frame) // c.FrameLength
        target = -q if target_frame < 0 else q  # Go integer division truncates toward zero
        target = max(0, min(target, len(self.samples)))
        self.sampleIdx = target
        self._buf, self._bufOff = b'', 0
        self._eof = target >= len(self.samples)
        return self.sampleIdx * c.FrameLength * _NS // c.SampleRate

    def _fill(self):
        idx = self.sampleIdx
        if not (self._ready is not None and self._ready_base <= idx < self._ready_base + self._ready_n):
            hi = min(len(self.samples), idx + self._window)
            out, nb, st = self.dec.decode_in_place(self._img_ptr, self._img_len, self._offs[idx:hi], self._sizes[idx:hi])
            # the arena is reused by the next window: keep this window's PCM
            self._ready = (out.copy(), nb, st)
            self._ready_n = hi - idx
            self._ready_base = idx
        out, nb, st = self._ready
        k = idx - self._ready_base
        if st[k] == ST_IO_TRUNCATED:  # io.ReadFull failure, decode.go:172-174
            raise IOError(f'reading sample {idx}: unexpected EOF')
        if st[k] != ST_OK:
            raise _packet_error(idx, int(st[k]))
        self._buf, self._bufOff = out[k, :nb[k]].tobytes(), 0
        self.sampleIdx += 1

    def Read(self, n: int) -> bytes:
        """io.Reader: up to n bytes; b'' means io.EOF (decode.go:127-190)."""
        out = bytearray()
        while len(out) < n:
            if self._bufOff < len(self._buf):
                take = min(n - len(out), len(self._buf) - self._bufOff)
                out += self._buf[self._bufOff:self._bufOff + take]
                self._bufOff += take
                continue
            if self._eof or self.sampleIdx >= len(self.samples):
                self._eof = True
                break
            try:
                self._fill()
            except Exception:
                if out:  # Go returns (total, err): hand out the bytes now, the error on the next call
                    break
                raise
        return bytes(out)

    def ReadAll(self) -> bytes:
        chunks = []
        while True:
            b = self.Read(1 << 24)
            if not b:
                return b''.join(chunks)
            chunks.append(b)


def NewDecoder(rs, device: int = 0, window: int = 2048) -> Decoder:
    return Decoder(rs, device, window)


@dataclass
class LoadedTrack:
    """One element of LoadTracks: samples [channels, frames] on the device and the PCMFormat, or the error."""
    samples: object = None  # torch.Tensor
    format: PCMFormat = None
    err: Exception = None


def LoadTracks(files, device: int = 0, dtype=None):
    """Many M4A files (bytes or file objects) as channel-planar CUDA tensors in one decode call: -> [LoadedTrack].
    Element t is what LoadTrack(files[t], device, dtype) returns (samples, format) or raises (err): the same values,
    shape, dtype and device, the same exception type, text and status. One bad file does not fail the others.

    The containers are parsed on the host; a track's packets from the first sample outside its file on are not
    decoded (that sample is its IOError). The decodable tracks are ordered by kernel config, their images and sample
    tables are uploaded through one pinned buffer in one copy, and one LibraryDecoder.DecodePlanar call decodes them.
    One [T, 3] array comes back: each track's frame total, first failing packet and its status word, reduced per track
    on the device. The samples of all tracks are views of one allocation."""
    import torch
    dev = torch.device('cuda', device)
    out = [LoadedTrack() for _ in files]
    todo = []  # (t, data, config, cookie, offsets, sizes, packets before the first one outside the file)
    for t, rs in enumerate(files):
        try:
            data, config, samples, cookie = _open_track(rs)
            st = _config_status(config)
            if st != ST_OK:
                raise _config_error(st, config)
            _planar_type(torch, dtype, (config.BitDepth,))
        except Exception as e:  # noqa: BLE001 -- the element's error, exactly what LoadTrack raises
            out[t].err = e
            continue
        n = len(samples)
        offs = np.array([o for o, _ in samples], dtype=np.uint64).reshape(n)
        sizes = np.array([z for _, z in samples], dtype=np.uint32).reshape(n)
        size = np.uint64(len(data))
        outside = (offs > size) | (sizes.astype(np.uint64) > size - np.minimum(offs, size))  # never handed to the kernel
        todo.append((t, data, config, cookie, offs, sizes, int(np.argmax(outside)) if outside.any() else n))
    if not todo:
        return out
    todo.sort(key=lambda x: (x[2].BitDepth, x[2].NumChannels, x[2].FrameLength, x[2].PB, x[2].MB, x[2].KB))
    # one pinned buffer, one copy: the images (each 16-byte aligned), then offsets i64 [N], sizes i32 [N], the row's
    # track i32 [N], the row's packet index in its track i32 [N], and each track's total in frame_start i64 [T]
    nt = len(todo)
    counts = np.array([x[6] for x in todo], dtype=np.int64)
    rows = int(counts.sum())
    bases = np.zeros(nt, dtype=np.int64)
    pos = 0
    for k, x in enumerate(todo):
        bases[k] = pos
        pos += (len(x[1]) + 15) // 16 * 16
    img = max(pos, 16)
    size16 = lambda b: (int(b) + 15) // 16 * 16  # noqa: E731
    at = [img]
    for b in (8 * rows, 4 * rows, 4 * rows, 4 * rows):
        at.append(size16(at[-1] + b))
    host = torch.empty(size16(at[-1] + 8 * nt), dtype=torch.uint8, pin_memory=True)
    h = host.numpy()
    first_row = np.concatenate([[0], np.cumsum(counts)[:-1]]).astype(np.int64)
    for k, x in enumerate(todo):
        h[bases[k]:bases[k] + len(x[1])] = np.frombuffer(x[1], dtype=np.uint8)
        a = first_row[k]
        h[at[0] + 8 * a:at[0] + 8 * (a + counts[k])].view(np.int64)[:] = x[4][:counts[k]].view(np.int64) + bases[k]
        h[at[1] + 4 * a:at[1] + 4 * (a + counts[k])].view(np.uint32)[:] = x[5][:counts[k]]
    h[at[2]:at[2] + 4 * rows].view(np.int32)[:] = np.repeat(np.arange(nt, dtype=np.int32), counts)
    h[at[3]:at[3] + 4 * rows].view(np.int32)[:] = np.arange(rows, dtype=np.int32) - np.repeat(first_row, counts).astype(np.int32)
    h[at[4]:at[4] + 8 * nt].view(np.int64)[:] = first_row + counts + np.arange(nt)
    lib_dec = LibraryDecoder((device,))
    try:
        with torch.cuda.device(dev):
            d = host.to(dev, non_blocking=True)
            d_offsets = d[at[0]:at[0] + 8 * rows].view(torch.int64)
            d_sizes = d[at[1]:at[1] + 4 * rows].view(torch.int32)
            track = d[at[2]:at[2] + 4 * rows].view(torch.int32).long()
            index = d[at[3]:at[3] + 4 * rows].view(torch.int32).long()
            totals_at = d[at[4]:at[4] + 8 * nt].view(torch.int64)
            pcm, frame_start, status, errors = lib_dec.DecodePlanar(d[:img], d_offsets, d_sizes, [x[3] for x in todo], counts,
                                                                    dtype, device)
            # per track, the first failing packet and its status in one key: index << 32 | status, minimum over the track
            none = torch.iinfo(torch.int64).max
            key = torch.where(status != 0, (index << 32) | (status.long() & 0xffffffff), none)
            first = torch.full((nt,), none, dtype=torch.int64, device=dev).scatter_reduce_(0, track, key, 'amin')
            info = torch.stack([frame_start[totals_at], first >> 32, first & 0xffffffff], 1).cpu().tolist()
    finally:
        lib_dec.close()
    for k, x in enumerate(todo):
        t, config, n, n_ok = x[0], x[2], len(x[4]), x[6]
        total, first_bad, first_status = info[k]
        if errors[k] is not None:
            out[t].err = errors[k]
        elif first_bad < n_ok:
            out[t].err = _packet_error(first_bad, first_status)
        elif n_ok < n:
            out[t].err = IOError(f'reading sample {n_ok}: unexpected EOF')  # io.ReadFull, decode.go:172-174
        else:
            out[t].samples = pcm[k][:, :total]
            out[t].format = PCMFormat(config.SampleRate, config.BitDepth, config.NumChannels)
    return out


def LoadTrack(rs, device: int = 0, dtype=None):
    """An M4A (bytes or a file object) as a channel-planar CUDA tensor: -> (samples [channels, frames] on cuda:device,
    PCMFormat). The samples are exactly what NewDecoder(rs).ReadAll() returns, reinterpreted as dtype (see
    PacketDecoder.DecodePlanar), and the errors are ReadAll's: ErrNoTrack, ErrConfig, ErrDecode for the first failing
    packet, IOError when a sample lies outside the file, whichever comes first in packet order.

    LoadTracks([rs], device, dtype)[0]: the file image and its sample table are uploaded once, the packets before the
    first sample outside the image are decoded in one call, and only the total frame count and the first failure come
    back to the host."""
    r = LoadTracks([rs], device, dtype)[0]
    if r.err is not None:
        raise r.err
    return r.samples, r.format
