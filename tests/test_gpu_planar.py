"""Channel-planar typed samples on the device (alacb200_decode_planar_device, PacketDecoder.DecodePlanar, LoadTrack).

Every comparison is exact: the expected samples are the oracle's interleaved PCM of the successful packets, read as
container values (oracle_lib.pcm_bytes_to_int), concatenated and transposed; F32 is that value times 2^-(8*bps-1).
"""
import io

import numpy as np
import pytest

import oracle_lib as ol
import synth_cases
from golden_io import load_fixtures
from m4a_writer import build_m4a
from signals import make_signal


@pytest.fixture(scope='module')
def pkg():
    from alac_b200_loader import load_package
    p = load_package()
    assert p.lib.alacb200_device_count() >= 1, 'no CUDA device: the product path has no CPU fallback'
    return p


def dtypes_for(bits):
    import torch
    return (torch.int16, torch.int32, torch.float32) if bits == 16 else (torch.int32, torch.float32)


def expected(ocfg, packed, offs, sizes):
    """Oracle -> (samples int64 [C, T], frame_start int64 [n + 1], status int32 [n])."""
    want, nb, st = ol.decode_batch(ocfg, packed, offs, sizes, nthreads=4)
    ch, bps = ocfg.num_channels, ocfg.bps()
    frame_start = np.concatenate([[0], np.cumsum(nb.astype(np.int64) // (ch * bps))])
    parts = [ol.pcm_bytes_to_int(want[i, :nb[i]].tobytes(), ocfg.bit_depth, ch) for i in range(len(sizes)) if st[i] == 0]
    x = np.concatenate(parts) if parts else np.zeros((0, ch), dtype=np.int64)
    return x.T, frame_start, st


def as_dtype(x, bits, dtype):
    """The container values x as the planar output of `dtype` (numpy)."""
    import torch
    if dtype == torch.float32:
        bps = {16: 2, 20: 3, 24: 3, 32: 4}[bits]
        return x.astype(np.float32) * np.float32(2.0 ** -(8 * bps - 1))
    return x.astype({torch.int16: np.int16, torch.int32: np.int32}[dtype])


def same(got, want):
    """Bit-for-bit equality of two arrays of one dtype (float compared as bits)."""
    got, want = np.ascontiguousarray(got), np.ascontiguousarray(want)
    if got.dtype == np.float32:
        got, want = got.view(np.int32), want.view(np.int32)
    return got.dtype == want.dtype and got.shape == want.shape and np.array_equal(got, want)


def to_device(packed, offs, sizes):
    import torch
    return (torch.from_numpy(np.ascontiguousarray(packed)).cuda(), torch.from_numpy(offs.view(np.int64)).cuda(),
            torch.from_numpy(sizes.view(np.int32)).cuda())


def check_planar(pkg, dec, ocfg, packets, name):
    """DecodePlanar for every sample type of the depth against the oracle; F32 == S32 * scale on the device."""
    import torch
    packed, offs, sizes = pkg.pack_packets(packets)
    x, want_fs, want_st = expected(ocfg, packed, offs, sizes)
    d = to_device(packed, offs, sizes)
    got = {}
    for dtype in dtypes_for(ocfg.bit_depth):
        samples, fs, st = dec.DecodePlanar(*d, dtype=dtype)
        assert samples.shape == (ocfg.num_channels, len(packets) * ocfg.frame_length), name
        assert np.array_equal(st.cpu().numpy(), want_st), (name, dtype)
        assert np.array_equal(fs.cpu().numpy(), want_fs), (name, dtype)
        total = int(want_fs[-1])
        assert same(samples[:, :total].cpu().numpy(), as_dtype(x, ocfg.bit_depth, dtype)), (name, dtype)
        got[dtype] = samples[:, :total]
    scale = 2.0 ** -(8 * ocfg.bps() - 1)
    assert torch.equal(got[torch.float32], got[torch.int32].float() * scale), name
    return want_st


def decoders(pkg):
    cache = {}

    def get(ocfg):
        key = bytes(ol.make_cookie(ocfg))
        if key not in cache:
            cache[key] = pkg.NewPacketDecoder(pkg.ParseMagicCookie(key), 0)
        return cache[key]
    return cache, get


def test_module_imports_without_torch():
    """The planar entry points import torch inside the call: loading the package must not."""
    import subprocess
    import sys
    code = ('import sys; from alac_b200_loader import load_package; p = load_package(); '
            'assert "torch" not in sys.modules; assert callable(p.LoadTrack) and hasattr(p.PacketDecoder, "DecodePlanar"); '
            'assert p.lib.alacb200_decode_planar_device(None, None, 0, None, None, 0, p.SAMPLES_F32, None, 0, None, None, None) == p.E_ARG')
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    subprocess.run([sys.executable, '-c', code], check=True, cwd=root)


@pytest.mark.gpu
def test_planar_golden_fixtures(pkg):
    """FFmpeg-encoded vectors: 1-8 channels, 16 / 24-bit, partial last packets."""
    cache, get = decoders(pkg)
    try:
        for name, fx in load_fixtures().items():
            st, ocfg = ol.parse_cookie(fx['cookie'])
            assert st == 0
            assert (check_planar(pkg, get(ocfg), ocfg, fx['packets'], name) == 0).all(), name
    finally:
        for d in cache.values():
            d.close()


@pytest.mark.gpu
def test_planar_exotic_shapes(pkg):
    """20 / 32-bit, shifted bytes 0-2, odd element orders, under-filled and partial packets."""
    cache, get = decoders(pkg)
    try:
        for name, ocfg, packets in synth_cases.exotic_cases():
            check_planar(pkg, get(ocfg), ocfg, packets, name)
    finally:
        for d in cache.values():
            d.close()


@pytest.mark.gpu
def test_planar_frame_lengths(pkg):
    """Frame lengths 1 ... 65536: tiles shorter than, equal to and many per packet; rows at every element alignment."""
    cache, get = decoders(pkg)
    try:
        for name, ocfg, packets in synth_cases.frame_length_cases():
            assert (check_planar(pkg, get(ocfg), ocfg, packets, name) == 0).all(), name
    finally:
        for d in cache.values():
            d.close()


@pytest.mark.gpu
def test_planar_failures_mid_batch(pkg):
    """Hostile packets between good ones: a failed packet takes no frames, the packets after it move up."""
    seen_fail = 0
    cache, get = decoders(pkg)
    try:
        for name, ocfg, bad in synth_cases.hostile_cases(max_per_seed=12):
            x = make_signal('silence_lsb', ocfg.num_channels, 5 * ocfg.frame_length + 300, ocfg.bit_depth, 48000, seed=len(bad))
            good = ol.encode_stream(ocfg, x)
            packets = good[:3] + bad[:len(bad) // 2] + good[3:5] + bad[len(bad) // 2:] + good[5:]
            st = check_planar(pkg, get(ocfg), ocfg, packets, name)
            seen_fail += int((st != 0).sum())
            assert (st[:3] == 0).all() and st[-1] == 0
    finally:
        for d in cache.values():
            d.close()
    assert seen_fail > 50


def raw_planar(pkg, dec, d, n, sample_type, out_ptr, stride, fs_ptr, st_ptr, stream=None):
    d_packed, d_off, d_sz = d
    return pkg.lib.alacb200_decode_planar_device(dec._h, d_packed.data_ptr(), d_packed.numel(), d_off.data_ptr(), d_sz.data_ptr(),
                                                 n, sample_type, out_ptr, stride, fs_ptr, st_ptr, stream)


@pytest.mark.gpu
def test_planar_channel_stride_and_unaligned_output(pkg):
    """channel_stride > n * frame_length (odd, so every channel row starts at another element alignment) and d_out one
    element past a 16-byte boundary: the samples are in place, frames past the total and the elements around the
    output keep their sentinel."""
    import torch
    for bits, ch, sample_type, dtype in ((24, 2, pkg.SAMPLES_S32, torch.int32), (24, 3, pkg.SAMPLES_F32, torch.float32),
                                         (16, 2, pkg.SAMPLES_S16, torch.int16), (16, 6, pkg.SAMPLES_F32, torch.float32)):
        ocfg = ol.Config.make(bit_depth=bits, num_channels=ch, sample_rate=48000)
        x = make_signal('music', ch, 4096 * 5 + 777, bits, 48000, seed=bits + ch)
        packets = ol.encode_stream(ocfg, x)
        packets.insert(2, b'\x80' + bytes(40))  # an unsupported element: fails, takes no frames
        packets.insert(4, ol.encode_packet(ocfg, x[:1001]))  # short packet in the middle: later packets start unaligned
        n = len(packets)
        packed, offs, sizes = pkg.pack_packets(packets)
        want, want_fs, want_st = expected(ocfg, packed, offs, sizes)
        assert want_st[2] != 0 and (np.delete(want_st, 2) == 0).all()
        dec = pkg.NewPacketDecoder(pkg.ParseMagicCookie(ol.make_cookie(ocfg)), 0)
        try:
            stride = n * 4096 + 37
            store = torch.int16 if dtype == torch.int16 else torch.int32
            sentinel = -12345
            buf = torch.full((ch * stride + 2,), sentinel, dtype=store, device='cuda')
            fs = torch.full((n + 1,), -1, dtype=torch.int64, device='cuda')
            st = torch.full((n,), -1, dtype=torch.int32, device='cuda')
            esz = buf.element_size()
            rc = raw_planar(pkg, dec, to_device(packed, offs, sizes), n, sample_type, buf.data_ptr() + esz, stride, fs.data_ptr(), st.data_ptr())
            assert rc == 0, pkg.lib.alacb200_last_error()
            torch.cuda.synchronize()
            assert np.array_equal(st.cpu().numpy(), want_st) and np.array_equal(fs.cpu().numpy(), want_fs)
            total = int(want_fs[-1])
            host = buf.cpu()
            assert int(host[0]) == sentinel and int(host[-1]) == sentinel
            rows = host[1:1 + ch * stride].view(ch, stride)
            got = rows[:, :total].view(dtype).numpy()
            assert same(got, as_dtype(want, bits, dtype)), (bits, ch, dtype)
            assert (rows[:, total:] == sentinel).all(), (bits, ch, dtype)
        finally:
            dec.close()


@pytest.mark.gpu
def test_planar_on_a_side_stream(pkg):
    """DecodePlanar enqueues on the current (non-default) stream and does not synchronise: the results are complete
    once that stream is."""
    import torch
    ocfg = ol.Config.make(bit_depth=24, num_channels=2, sample_rate=96000)
    x = make_signal('bench', 2, 4096 * 300 + 55, 24, 96000, seed=77)
    packets = ol.encode_stream(ocfg, x)
    packed, offs, sizes = pkg.pack_packets(packets)
    d = to_device(packed, offs, sizes)
    torch.cuda.synchronize()
    dec = pkg.NewPacketDecoder(pkg.ParseMagicCookie(ol.make_cookie(ocfg)), 0)
    try:
        side = torch.cuda.Stream()
        with torch.cuda.stream(side):
            samples, fs, st = dec.DecodePlanar(*d)
            samples2, _, _ = dec.DecodePlanar(*d, dtype=torch.int32)  # the same decoder again on the same stream
        side.synchronize()
        total = len(x)
        assert (st.cpu() == 0).all() and int(fs[-1]) == total
        assert same(samples[:, :total].cpu().numpy(), as_dtype(x.T, 24, torch.float32))
        assert same(samples2[:, :total].cpu().numpy(), x.T.astype(np.int32))
        # and back on the default stream: the decoder's scratch follows the caller's stream
        samples3, _, _ = dec.DecodePlanar(*d, dtype=torch.int32)
        assert torch.equal(samples3[:, :total], samples2[:, :total])
    finally:
        dec.close()


@pytest.mark.gpu
def test_planar_argument_errors(pkg):
    """ALACB200_E_ARG: unknown sample type, S16 on a 24-bit stream, NULL pointers, a channel stride under
    n * frame_length, d_out not aligned to its element, d_packed not 16-byte aligned. n == 0 writes frame_start[0] = 0."""
    import torch
    ocfg = ol.Config.make(bit_depth=24, num_channels=2, sample_rate=48000)
    packets = ol.encode_stream(ocfg, make_signal('music', 2, 4096 * 3, 24, 48000, seed=3))
    n = len(packets)
    packed, offs, sizes = pkg.pack_packets(packets)
    d = to_device(packed, offs, sizes)
    dec = pkg.NewPacketDecoder(pkg.ParseMagicCookie(ol.make_cookie(ocfg)), 0)
    try:
        out = torch.zeros(2 * n * 4096 + 8, dtype=torch.int32, device='cuda')
        fs = torch.full((n + 1,), -1, dtype=torch.int64, device='cuda')
        st = torch.zeros(n, dtype=torch.int32, device='cuda')
        o, f, s = out.data_ptr(), fs.data_ptr(), st.data_ptr()
        stride = n * 4096
        E = pkg.E_ARG
        assert raw_planar(pkg, dec, d, n, 0, o, stride, f, s) == E
        assert raw_planar(pkg, dec, d, n, 4, o, stride, f, s) == E
        assert raw_planar(pkg, dec, d, n, pkg.SAMPLES_S16, o, stride, f, s) == E
        assert raw_planar(pkg, dec, d, n, pkg.SAMPLES_F32, None, stride, f, s) == E
        assert raw_planar(pkg, dec, d, n, pkg.SAMPLES_F32, o, stride, None, s) == E
        assert raw_planar(pkg, dec, d, n, pkg.SAMPLES_F32, o, stride, f, None) == E
        d_packed, d_off, d_sz = d
        call = pkg.lib.alacb200_decode_planar_device
        assert call(dec._h, None, d_packed.numel(), d_off.data_ptr(), d_sz.data_ptr(), n, pkg.SAMPLES_F32, o, stride, f, s, None) == E
        assert call(dec._h, d_packed.data_ptr(), d_packed.numel(), None, d_sz.data_ptr(), n, pkg.SAMPLES_F32, o, stride, f, s, None) == E
        assert call(dec._h, d_packed.data_ptr(), d_packed.numel(), d_off.data_ptr(), None, n, pkg.SAMPLES_F32, o, stride, f, s, None) == E
        assert call(None, d_packed.data_ptr(), d_packed.numel(), d_off.data_ptr(), d_sz.data_ptr(), n, pkg.SAMPLES_F32, o, stride, f, s, None) == E
        assert call(dec._h, d_packed.data_ptr() + 8, d_packed.numel() - 16, d_off.data_ptr(), d_sz.data_ptr(), n, pkg.SAMPLES_F32, o, stride, f, s, None) == E
        assert raw_planar(pkg, dec, d, n, pkg.SAMPLES_F32, o, stride - 1, f, s) == E
        assert raw_planar(pkg, dec, d, n, pkg.SAMPLES_F32, o + 2, stride, f, s) == E
        assert raw_planar(pkg, dec, d, n, pkg.SAMPLES_S32, o + 1, stride, f, s) == E
        with pytest.raises(ValueError):
            dec.DecodePlanar(*d, dtype=torch.int16)
        with pytest.raises(ValueError):
            dec.DecodePlanar(*d, dtype=torch.float64)
        torch.cuda.synchronize()
        assert (fs.cpu() == -1).all() and (out.cpu() == 0).all()  # nothing was enqueued
        assert raw_planar(pkg, dec, d, 0, pkg.SAMPLES_F32, None, 0, f, None) == 0
        torch.cuda.synchronize()
        assert int(fs[0]) == 0 and (fs[1:].cpu() == -1).all()
        # the decoder still works after the rejected calls
        assert raw_planar(pkg, dec, d, n, pkg.SAMPLES_S32, o, stride, f, s) == 0
        torch.cuda.synchronize()
        assert (st.cpu() == 0).all() and int(fs[n]) == n * 4096
        samples, fs2, _ = dec.DecodePlanar(d[0], d[1][:0], d[2][:0])
        assert samples.shape == (2, 0) and fs2.cpu().tolist() == [0]
    finally:
        dec.close()


def read_all_samples(pkg, data, dtype, bits, ch):
    """What LoadTrack must return: NewDecoder(data).ReadAll() reinterpreted as [channels, frames] of dtype."""
    dec = pkg.NewDecoder(data)
    try:
        pcm = dec.ReadAll()
    finally:
        dec.close()
    return as_dtype(ol.pcm_bytes_to_int(pcm, bits, ch).T, bits, dtype)


@pytest.mark.gpu
def test_load_track_c1_full_size(pkg):
    """BASELINE configs[0] at full size (60 s, 646 packets, the last one short), moov after and before mdat, from bytes
    and from a file object: for every sample type, LoadTrack == NewDecoder(...).ReadAll() reinterpreted."""
    import bench
    import torch
    wl = bench.build_workload('c1', seed=1, threads=bench.host_cores())
    packets = [bytes(wl['packed'][int(o):int(o) + int(z)]) for o, z in zip(wl['offsets'], wl['sizes'])]
    for kw in (dict(samples_per_chunk=9), dict(moov_first=True)):
        data, _ = build_m4a(wl['cookie'], packets, last_frames=wl['frames'] % 4096, **kw)
        for dtype in dtypes_for(16):
            got, fmt = pkg.LoadTrack(data, 0, dtype)
            assert fmt == pkg.PCMFormat(44100, 16, 2)
            assert got.is_cuda and got.dtype == dtype and got.shape == (2, wl['frames'])
            assert same(got.cpu().numpy(), read_all_samples(pkg, data, dtype, 16, 2)), (kw, dtype)
        got, _ = pkg.LoadTrack(io.BytesIO(data), dtype=torch.int32)
        assert same(got.cpu().numpy(), read_all_samples(pkg, data, torch.int32, 16, 2))


def error_of(f):
    try:
        f()
    except Exception as e:  # noqa: BLE001 -- the exception itself is the result
        return type(e), str(e), getattr(e, 'status', None)
    return None


@pytest.mark.gpu
def test_load_track_errors_match_read_all(pkg):
    """LoadTrack raises what ReadAll raises, type and text: a sample past EOF, a corrupted packet, the first of the two in
    packet order, no track, a bad cookie; and a file that decodes still loads."""
    import torch
    ocfg = ol.Config.make(bit_depth=16, num_channels=2, sample_rate=44100)
    x = make_signal('music', 2, 4096 * 10 + 500, 16, 44100, seed=12)
    packets = ol.encode_stream(ocfg, x)
    data, samples = build_m4a(ol.make_cookie(ocfg), packets, last_frames=500, moov_first=True)

    def corrupt(d, k):  # packet k keeps its headers, its entropy-coded data becomes 0xff: ErrDecode (bitstream overrun) at k
        d = bytearray(d)
        off, size = samples[k]
        d[off + 8:off + size] = b'\xff' * (size - 8)
        return bytes(d)

    def cut(d, k):  # the file ends in the middle of packet k
        off, size = samples[k]
        return d[:off + size // 2]

    cases = {
        'truncated': cut(data, 6),
        'corrupted': corrupt(data, 3),
        'corrupted before truncated': cut(corrupt(data, 3), 7),
        'truncated before corrupted': cut(corrupt(data, 8), 5),
        'no track': b'\0\0\0\x10free' + bytes(64),
        'bad cookie': build_m4a(ol.make_cookie(ocfg, 1)[:30], packets)[0],
    }
    kinds = {}
    for name, d in cases.items():
        want = error_of(lambda: pkg.NewDecoder(d).ReadAll())
        assert want is not None, name
        kinds[name] = want[0]
        for dtype in (torch.float32, torch.int16):
            assert error_of(lambda: pkg.LoadTrack(d, dtype=dtype)) == want, (name, dtype)
    assert issubclass(kinds['truncated'], IOError) and kinds['corrupted'] is pkg.ErrDecode
    assert kinds['corrupted before truncated'] is pkg.ErrDecode and issubclass(kinds['truncated before corrupted'], IOError)
    assert kinds['no track'] is pkg.ErrNoTrack and kinds['bad cookie'] is pkg.ErrConfig
    got, _ = pkg.LoadTrack(data, dtype=torch.int16)
    assert same(got.cpu().numpy(), x.T.astype(np.int16))


@pytest.mark.gpu
def test_planar_full_size_c3_matches_interleaved(pkg):
    """BASELINE configs[2] at full size (168 750 packets, 24-bit stereo): F32 planar output == the interleaved device
    path's PCM for the same packets, converted to float on the GPU with torch."""
    import bench
    import torch
    wl = bench.build_workload('c3', seed=3, threads=bench.host_cores())
    n = len(wl['sizes'])
    assert n == 168750
    d = to_device(wl['packed'], wl['offsets'], wl['sizes'])
    dec = pkg.NewPacketDecoder(pkg.ParseMagicCookie(wl['cookie']))
    try:
        fb = dec.frame_bytes
        pcm = torch.empty(n * fb, dtype=torch.uint8, device='cuda')
        nb = torch.empty(n, dtype=torch.int32, device='cuda')
        st = torch.empty(n, dtype=torch.int32, device='cuda')
        rc = pkg.lib.alacb200_decode_packets_device(dec._h, d[0].data_ptr(), d[0].numel(), d[1].data_ptr(), d[2].data_ptr(), n,
                                                    pcm.data_ptr(), fb, nb.data_ptr(), st.data_ptr(), None)
        assert rc == 0
        samples, fs, pst = dec.DecodePlanar(*d)
        torch.cuda.synchronize()
        assert (st == 0).all() and (pst == 0).all()
        frames = nb.long() // 6
        assert torch.equal(fs[1:], torch.cumsum(frames, 0)) and int(fs[0]) == 0 and int(fs[n]) == wl['frames']
        step = 16384
        for a in range(0, n, step):
            b = min(n, a + step)
            f0, f1 = int(fs[a]), int(fs[b])
            raw = pcm[a * fb:a * fb + (f1 - f0) * 6].view(-1, 3).int()  # every packet but the last is full: contiguous
            v = raw[:, 0] | (raw[:, 1] << 8) | (raw[:, 2].to(torch.uint8).view(torch.int8).int() << 16)
            want = (v.float() * 2.0 ** -23).view(-1, 2).t()
            assert torch.equal(samples[:, f0:f1], want), (a, b)
    finally:
        dec.close()
