"""Many tracks in one planar call (alacb200_library_decode_planar_device, LibraryDecoder.DecodePlanar, LoadTracks).

Every comparison is exact. LoadTracks is checked element by element against LoadTrack of the same file and against
NewDecoder(...).ReadAll(); the raw entry point against the oracle's interleaved PCM read as container values.
"""
import io
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle_lib as ol
import synth_cases
from golden_io import load_fixtures
from m4a_writer import build_m4a
from signals import make_signal

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope='module')
def pkg():
    from alac_b200_loader import load_package
    p = load_package()
    assert p.lib.alacb200_device_count() >= 1, 'no CUDA device: the product path has no CPU fallback'
    return p


def same(got, want):
    """Bit-for-bit equality of two arrays of one dtype (float compared as bits)."""
    got, want = np.ascontiguousarray(got), np.ascontiguousarray(want)
    if got.dtype == np.float32:
        got, want = got.view(np.int32), want.view(np.int32)
    return got.dtype == want.dtype and got.shape == want.shape and np.array_equal(got, want)


def as_dtype(x, bits, dtype):
    """Container values x as the planar output of `dtype` (numpy)."""
    import torch
    if dtype == torch.float32:
        return x.astype(np.float32) * np.float32(2.0 ** -(8 * {16: 2, 20: 3, 24: 3, 32: 4}[bits] - 1))
    return x.astype({torch.int16: np.int16, torch.int32: np.int32}[dtype])


def outcome(f):
    """-> ('ok', samples, format) or ('err', type, str, status) of a LoadTrack call."""
    try:
        samples, fmt = f()
    except Exception as e:  # noqa: BLE001 -- the exception itself is the result
        return ('err', type(e), str(e), getattr(e, 'status', None))
    return ('ok', samples, fmt)


def check_element(pkg, got, want, name):
    """A LoadedTrack equals LoadTrack's outcome: the same error, or the same samples (values, shape, dtype, device)."""
    if want[0] == 'err':
        assert got.err is not None and got.samples is None, name
        assert (type(got.err), str(got.err), getattr(got.err, 'status', None)) == want[1:], name
        return
    assert got.err is None, (name, got.err)
    samples, fmt = want[1], want[2]
    assert got.format == fmt, name
    assert got.samples.dtype == samples.dtype and got.samples.device == samples.device, name
    assert same(got.samples.cpu().numpy(), samples.cpu().numpy()), name


def read_all(pkg, data, dtype):
    """NewDecoder(data).ReadAll() as [channels, frames] of dtype."""
    dec = pkg.NewDecoder(data)
    try:
        pcm = dec.ReadAll()
        fmt = dec.Format()
    finally:
        dec.close()
    return as_dtype(ol.pcm_bytes_to_int(pcm, fmt.BitDepth, fmt.Channels).T, fmt.BitDepth, dtype)


def mixed_files():
    """(name, file bytes) of the golden fixtures (1-8 channels, 16 / 24-bit, partial last packets) and synthetic 20 and
    32-bit tracks, interleaved so that consecutive files have different configs."""
    by_cfg = {}
    for name, fx in load_fixtures().items():
        st, ocfg = ol.parse_cookie(fx['cookie'])
        assert st == 0
        data, _ = build_m4a(fx['cookie'], fx['packets'], channels=ocfg.num_channels, bits=ocfg.bit_depth)
        by_cfg.setdefault((ocfg.bit_depth, ocfg.num_channels, ocfg.frame_length), []).append((name, data))
    for bits, ch, seed in ((20, 2, 5), (32, 1, 6), (20, 6, 7), (32, 2, 8)):
        ocfg = ol.Config.make(bit_depth=bits, num_channels=ch, sample_rate=48000)
        x = make_signal('music', ch, 4096 * 3 + 333 * seed, bits, 48000, seed=seed)
        data, _ = build_m4a(ol.make_cookie(ocfg), ol.encode_stream(ocfg, x), channels=ch, bits=bits)
        by_cfg.setdefault((bits, ch, 4096), []).append((f'synth{bits}x{ch}', data))
    groups = list(by_cfg.values())
    out = []
    while any(groups):
        for g in groups:
            if g:
                out.append(g.pop(0))
    return out


def test_imports_without_torch_and_null_library():
    """LoadTracks and the new entry point are reachable without torch; a NULL library is ALACB200_E_ARG."""
    code = ('import sys; from alac_b200_loader import load_package; p = load_package(); '
            'assert "torch" not in sys.modules; assert callable(p.LoadTracks) and hasattr(p.LibraryDecoder, "DecodePlanar"); '
            'assert p.lib.alacb200_library_decode_planar_device(None, 0, None, 0, None, None, None, 0, p.SAMPLES_F32, None, None, None) == p.E_ARG; '
            'assert "torch" not in sys.modules')
    subprocess.run([sys.executable, '-c', code], check=True, cwd=ROOT)


@pytest.mark.gpu
def test_mixed_batch_equals_load_track(pkg):
    """Every dtype: each element of one LoadTracks call over alternating configs (some files as file objects) equals
    LoadTrack of the same file and ReadAll reinterpreted; with int16 the non-16-bit files carry LoadTrack's ValueError."""
    import torch
    files = mixed_files()
    assert len({n for n, _ in files}) == len(files) >= 10
    for dtype in (torch.float32, torch.int32, torch.int16):
        inputs = [io.BytesIO(d) if k % 3 == 1 else d for k, (_, d) in enumerate(files)]
        got = pkg.LoadTracks(inputs, 0, dtype)
        assert len(got) == len(files)
        n_ok = 0
        for (name, data), g in zip(files, got):
            want = outcome(lambda: pkg.LoadTrack(io.BytesIO(data), 0, dtype))
            check_element(pkg, g, want, (name, dtype))
            if want[0] == 'ok':
                n_ok += 1
                assert same(g.samples.cpu().numpy(), read_all(pkg, data, dtype)), (name, dtype)
            else:
                assert dtype == torch.int16 and want[1] is ValueError, (name, want)
        assert n_ok >= 3


def error_files():
    """(name, file bytes) of files LoadTrack fails on, and good files of two configs."""
    ocfg = ol.Config.make(bit_depth=16, num_channels=2, sample_rate=44100)
    x = make_signal('music', 2, 4096 * 10 + 500, 16, 44100, seed=12)
    packets = ol.encode_stream(ocfg, x)
    data, samples = build_m4a(ol.make_cookie(ocfg), packets, last_frames=500, moov_first=True)

    def corrupt(d, k):  # packet k's entropy-coded data becomes 0xff: ErrDecode (bitstream overrun) at k
        d = bytearray(d)
        off, size = samples[k]
        d[off + 8:off + size] = b'\xff' * (size - 8)
        return bytes(d)

    def cut(d, k):  # the file ends in the middle of packet k
        off, size = samples[k]
        return d[:off + size // 2]

    bad = {
        'truncated': cut(data, 6),
        'corrupted': corrupt(data, 3),
        'corrupted before truncated': cut(corrupt(data, 3), 7),
        'truncated before corrupted': cut(corrupt(data, 8), 5),
        'no track': b'\0\0\0\x10free' + bytes(64),
        'bad cookie': build_m4a(ol.make_cookie(ocfg, 1)[:30], packets)[0],
        'unsupported depth': build_m4a(ol.make_cookie(ol.Config.make(bit_depth=12, num_channels=2, sample_rate=44100)), packets)[0],
        'zero samples': build_m4a(ol.make_cookie(ocfg), [])[0],
    }
    o24 = ol.Config.make(bit_depth=24, num_channels=2, sample_rate=48000)
    good = [('good16', data)]
    for seed in (1, 2):
        y = make_signal('music', 2, 4096 * 4 + 77 * seed, 24, 48000, seed=seed)
        good.append((f'good24_{seed}', build_m4a(ol.make_cookie(o24), ol.encode_stream(o24, y), bits=24, rate=48000)[0]))
    return bad, good


@pytest.mark.gpu
def test_failures_do_not_leak(pkg):
    """Each failing file between good files of different configs gets LoadTrack's error (type, text, status), and
    every good file is still exact."""
    import torch
    bad, good = error_files()
    files = []
    for k, item in enumerate(bad.items()):
        files += [good[k % len(good)], item]
    files.append(good[0])
    for dtype in (torch.float32, torch.int16):
        got = pkg.LoadTracks([d for _, d in files], 0, dtype)
        for (name, data), g in zip(files, got):
            want = outcome(lambda: pkg.LoadTrack(data, 0, dtype))
            check_element(pkg, g, want, (name, dtype))
            if name in bad and name != 'zero samples':
                assert want[0] == 'err', name
                if name != 'unsupported depth':  # ReadAll raises the same error
                    try:
                        pkg.NewDecoder(data).ReadAll()
                        raise AssertionError(name)
                    except Exception as e:  # noqa: BLE001
                        assert (type(e), str(e), getattr(e, 'status', None)) == want[1:], name
            elif want[0] == 'ok':
                assert same(g.samples.cpu().numpy(), read_all(pkg, data, dtype)), (name, dtype)
    zero = got[[n for n, _ in files].index('zero samples')]
    assert zero.err is not None or zero.samples.shape[1] == 0


# ---- the raw entry point ------------------------------------------------------------------------------------------

def track_packets(bits, ch, frames, seed, extra_bad=False):
    ocfg = ol.Config.make(bit_depth=bits, num_channels=ch, sample_rate=48000)
    packets = ol.encode_stream(ocfg, make_signal('music', ch, frames, bits, 48000, seed=seed))
    if extra_bad:
        packets.insert(1, b'\x80' + bytes(40))  # an unsupported element: fails, takes no frames
    return ocfg, packets


def oracle_track(ocfg, packets):
    """-> (container values int64 [C, T], frame starts int64 [n + 1], status [n])."""
    packed, offs, sizes = ol.pack(packets)
    want, nb, st = ol.decode_batch(ocfg, packed, offs, sizes, nthreads=4)
    ch, bps = ocfg.num_channels, ocfg.bps()
    fs = np.concatenate([[0], np.cumsum(nb.astype(np.int64) // (ch * bps))])
    parts = [ol.pcm_bytes_to_int(want[i, :nb[i]].tobytes(), ocfg.bit_depth, ch) for i in range(len(packets)) if st[i] == 0]
    x = np.concatenate(parts) if parts else np.zeros((0, ch), dtype=np.int64)
    return x.T, fs, st


class RawBatch:
    """Tracks (ocfg, packets) in one packet table on the device, and ctypes descriptors for the raw call."""

    def __init__(self, pkg, tracks):
        import torch
        self.pkg, self.tracks = pkg, tracks
        allp = [p for _, ps in tracks for p in ps]
        packed, offs, sizes = pkg.pack_packets(allp)
        self.rows = len(allp)
        self.d = (torch.from_numpy(packed).cuda(), torch.from_numpy(offs.view(np.int64)).cuda(),
                  torch.from_numpy(sizes.view(np.int32)).cuda())
        self.cookies = [np.frombuffer(ol.make_cookie(c), dtype=np.uint8) for c, _ in tracks]
        self.want = [oracle_track(c, ps) for c, ps in tracks]

    def descs(self, outs, strides):
        pkg = self.pkg
        descs = (pkg.PlanarTrackDesc * max(1, len(self.tracks)))()
        for t, (_, ps) in enumerate(self.tracks):
            descs[t].cookie, descs[t].cookie_len = self.cookies[t].ctypes.data, len(self.cookies[t])
            descs[t].n, descs[t].d_out, descs[t].channel_stride = len(ps), outs[t], strides[t]
        return descs

    def call(self, descs, sample_type, fs, st, stream=None, packed=None, ntracks=None, device=0, lib_h=None):
        p, o, z = self.d
        return self.pkg.lib.alacb200_library_decode_planar_device(
            lib_h, device, p.data_ptr() if packed is None else packed, p.numel(), o.data_ptr(), z.data_ptr(), descs,
            len(self.tracks) if ntracks is None else ntracks, sample_type, fs, st, stream)


def sentinel_outputs(batch, dtype, pad=37):
    """Per track a sentinel-filled buffer; d_out one element in (never 16-byte aligned), channel_stride n*FL + pad."""
    import torch
    store = torch.int16 if dtype == torch.int16 else torch.int32
    bufs, outs, strides = [], [], []
    for c, ps in batch.tracks:
        stride = len(ps) * c.frame_length + pad
        b = torch.full((c.num_channels * stride + 2,), -12345, dtype=store, device='cuda')
        bufs.append(b)
        outs.append(b.data_ptr() + b.element_size())
        strides.append(stride)
    return bufs, outs, strides


def check_outputs(batch, bufs, strides, dtype, fs, st):
    import torch
    fs, st = fs.cpu().numpy(), st.cpu().numpy()
    row = 0
    for t, (c, ps) in enumerate(batch.tracks):
        x, want_fs, want_st = batch.want[t]
        n = len(ps)
        assert np.array_equal(st[row:row + n], want_st), t
        assert np.array_equal(fs[row + t:row + t + n + 1], want_fs), t
        total = int(want_fs[-1])
        host = bufs[t].cpu()
        assert int(host[0]) == -12345 and int(host[-1]) == -12345, t
        rows = host[1:1 + c.num_channels * strides[t]].view(c.num_channels, strides[t])
        assert same(rows[:, :total].view(dtype).numpy(), as_dtype(x, c.bit_depth, dtype)), (t, dtype)
        assert (rows[:, total:] == -12345).all(), t
        row += n
    assert row == batch.rows and len(fs) == batch.rows + len(batch.tracks)
    torch.cuda.synchronize()


def abab(pkg):
    a1 = track_packets(24, 2, 4096 * 5 + 100, 1, extra_bad=True)
    b1 = track_packets(16, 3, 4096 * 3 + 7, 2)
    a2 = track_packets(24, 2, 4096 * 2 + 1, 3)
    b2 = track_packets(16, 3, 4096 * 4, 4, extra_bad=True)
    return RawBatch(pkg, [a1, b1, a2, b2])


@pytest.mark.gpu
def test_raw_ungrouped_strided_unaligned(pkg):
    """Configs A, B, A, B (four runs), a failing packet in two tracks, channel_stride larger than needed and d_out at an
    odd element offset: the samples are in place and every sentinel around and between the rows is untouched; then the
    same on a side stream."""
    import torch
    batch = abab(pkg)
    libd = pkg.NewLibraryDecoder((0,))
    try:
        for sample_type, dtype in ((pkg.SAMPLES_S32, torch.int32), (pkg.SAMPLES_F32, torch.float32)):
            for side in (False, True):
                bufs, outs, strides = sentinel_outputs(batch, dtype)
                fs = torch.full((batch.rows + 4,), -1, dtype=torch.int64, device='cuda')
                st = torch.full((batch.rows,), -1, dtype=torch.int32, device='cuda')
                descs = batch.descs(outs, strides)
                torch.cuda.synchronize()
                if side:
                    stream = torch.cuda.Stream()
                    with torch.cuda.stream(stream):
                        rc = batch.call(descs, sample_type, fs.data_ptr(), st.data_ptr(), stream.cuda_stream, lib_h=libd._h)
                    stream.synchronize()
                else:
                    rc = batch.call(descs, sample_type, fs.data_ptr(), st.data_ptr(), lib_h=libd._h)
                    torch.cuda.synchronize()
                assert rc == 0, pkg.lib.alacb200_last_error()
                assert all(descs[t].result == 0 and descs[t].track_status == 0 for t in range(4))
                assert descs[1].config.BitDepth == 16 and descs[1].config.NumChannels == 3
                check_outputs(batch, bufs, strides, dtype, fs, st)
    finally:
        libd.close()


@pytest.mark.gpu
def test_raw_config_failure_is_per_track(pkg):
    """A track with a bad cookie between good ones: E_CONFIG with its status, its rows carry that status, its frame starts
    are 0, its output is untouched; the others decode. LibraryDecoder.DecodePlanar reports DecodeTracks' error."""
    import torch
    batch = abab(pkg)
    batch.cookies[2] = batch.cookies[2][:20]  # too short: ST_INVALID_COOKIE
    libd = pkg.NewLibraryDecoder((0,))
    try:
        bufs, outs, strides = sentinel_outputs(batch, torch.int32)
        fs = torch.full((batch.rows + 4,), -1, dtype=torch.int64, device='cuda')
        st = torch.full((batch.rows,), -1, dtype=torch.int32, device='cuda')
        descs = batch.descs(outs, strides)
        assert batch.call(descs, pkg.SAMPLES_S32, fs.data_ptr(), st.data_ptr(), lib_h=libd._h) == 0
        torch.cuda.synchronize()
        assert descs[2].result == pkg.E_CONFIG and descs[2].track_status == pkg.ST_INVALID_COOKIE
        counts = [len(ps) for _, ps in batch.tracks]
        starts = np.concatenate([[0], np.cumsum(counts)])
        r0, n2 = int(starts[2]), counts[2]
        assert (st[r0:r0 + n2].cpu() == pkg.ST_INVALID_COOKIE).all()
        assert (fs[r0 + 2:r0 + 2 + n2 + 1].cpu() == 0).all()
        assert (bufs[2].cpu() == -12345).all()
        for t in (0, 1, 3):
            x, want_fs, want_st = batch.want[t]
            a, n = int(starts[t]), counts[t]
            assert np.array_equal(st[a:a + n].cpu().numpy(), want_st) and np.array_equal(fs[a + t:a + t + n + 1].cpu().numpy(), want_fs)
            c = batch.tracks[t][0]
            rows = bufs[t].cpu()[1:1 + c.num_channels * strides[t]].view(c.num_channels, strides[t])
            assert same(rows[:, :int(want_fs[-1])].numpy(), x.astype(np.int32)), t
            assert (rows[:, int(want_fs[-1]):] == -12345).all(), t
        cookies = [c.tobytes() for c in batch.cookies]
        samples, fs2, st2, errs = libd.DecodePlanar(*batch.d, cookies, counts, dtype=torch.int32)
        torch.cuda.synchronize()
        assert samples[2] is None and samples[0] is not None
        want_err = pkg.error_from_status(pkg.ST_INVALID_COOKIE)
        assert type(errs[2]) is type(want_err) and str(errs[2]) == str(want_err) and errs[2].status == want_err.status
        assert torch.equal(fs2, fs) and torch.equal(st2, st)
    finally:
        libd.close()


@pytest.mark.gpu
def test_raw_argument_errors_and_empty(pkg):
    """ALACB200_E_ARG before anything is enqueued: unknown sample type, S16 with a 24-bit track, a channel stride too
    small, a misaligned d_out or d_packed, NULL pointers, a device not in the library. ntracks == 0 and all-zero n
    write only the frame starts, all 0."""
    import torch
    batch = abab(pkg)
    libd = pkg.NewLibraryDecoder((0,))
    try:
        bufs, outs, strides = sentinel_outputs(batch, torch.int32, pad=0)
        fs = torch.full((batch.rows + 4,), -1, dtype=torch.int64, device='cuda')
        st = torch.full((batch.rows,), -1, dtype=torch.int32, device='cuda')
        f, s, h = fs.data_ptr(), st.data_ptr(), libd._h
        E = pkg.E_ARG

        def call(outs=outs, strides=strides, sample_type=pkg.SAMPLES_S32, **kw):
            return batch.call(batch.descs(outs, strides), sample_type, kw.pop('fs', f), kw.pop('st', s), lib_h=kw.pop('lib_h', h), **kw)
        assert call(sample_type=0) == E and call(sample_type=4) == E
        assert call(sample_type=pkg.SAMPLES_S16) == E
        assert call(strides=[strides[0] - 1] + strides[1:]) == E
        assert call(outs=outs[:3] + [outs[3] + 1]) == E
        assert call(outs=outs[:1] + [None] + outs[2:]) == E
        assert call(packed=batch.d[0].data_ptr() + 8) == E
        assert call(fs=None) == E and call(st=None) == E and call(lib_h=None) == E
        assert call(device=1) == E and call(device=-1) == E
        p, o, z = batch.d
        descs = batch.descs(outs, strides)
        for args in ((None, o.data_ptr(), z.data_ptr()), (p.data_ptr(), None, z.data_ptr()), (p.data_ptr(), o.data_ptr(), None)):
            assert pkg.lib.alacb200_library_decode_planar_device(h, 0, args[0], p.numel(), args[1], args[2], descs, 4, pkg.SAMPLES_S32,
                                                                 f, s, None) == E
        assert pkg.lib.alacb200_library_decode_planar_device(h, 0, None, 0, None, None, None, 1, pkg.SAMPLES_S32, f, s, None) == E
        torch.cuda.synchronize()
        assert (fs.cpu() == -1).all() and (st.cpu() == -1).all() and all((b.cpu() == -12345).all() for b in bufs)
        # empty: no tracks, then four tracks without rows (one with a bad cookie)
        assert pkg.lib.alacb200_library_decode_planar_device(h, 0, None, 0, None, None, None, 0, pkg.SAMPLES_F32, None, None, None) == 0
        empty = RawBatch.__new__(RawBatch)
        empty.pkg, empty.tracks, empty.rows = pkg, [(c, []) for c, _ in batch.tracks], 0
        empty.cookies = batch.cookies[:3] + [batch.cookies[3][:10]]
        descs = empty.descs([None] * 4, [0] * 4)
        assert pkg.lib.alacb200_library_decode_planar_device(h, 0, None, 0, None, None, descs, 4, pkg.SAMPLES_F32, f, None, None) == 0
        torch.cuda.synchronize()
        assert fs[:4].cpu().tolist() == [0, 0, 0, 0] and (fs[4:].cpu() == -1).all()
        assert descs[3].result == pkg.E_CONFIG and descs[0].result == 0
        # and the library still decodes
        assert call() == 0
        torch.cuda.synchronize()
        check_outputs(batch, bufs, strides, torch.int32, fs, st)
    finally:
        libd.close()


@pytest.mark.gpu
def test_one_decode_launch_per_config(pkg):
    """torch.profiler: LoadTracks of 8 files of two configs launches the decode kernel twice; the raw call on the
    ungrouped A, B, A, B table launches it four times."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    files = []
    for k in range(8):
        bits = 16 if k % 2 else 24
        ocfg = ol.Config.make(bit_depth=bits, num_channels=2, sample_rate=44100)
        x = make_signal('music', 2, 4096 * (3 + k) + 11, bits, 44100, seed=40 + k)
        files.append(build_m4a(ol.make_cookie(ocfg), ol.encode_stream(ocfg, x), bits=bits)[0])
    pkg.LoadTracks(files)  # warm up
    batch = abab(pkg)
    libd = pkg.NewLibraryDecoder((0,))
    try:
        counts = [len(ps) for _, ps in batch.tracks]
        torch.cuda.synchronize()

        def launches(f):
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                f()
                torch.cuda.synchronize()
            names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
            return sum('alac_decode_kernel' in n for n in names), sum('alac_planar_kernel' in n for n in names)
        got = launches(lambda: pkg.LoadTracks(files))
        assert got == (2, 2), got
        got = launches(lambda: libd.DecodePlanar(*batch.d, [c.tobytes() for c in batch.cookies], counts))
        assert got == (4, 4), got
    finally:
        libd.close()


@pytest.mark.gpu
def test_library_batch_full_size(pkg):
    """bench.py's library batch (32 tracks of 3 min, 16- and 24-bit alternating) as M4A files through LoadTracks, F32
    and S32: equal to LibraryDecoder.DecodeTracks' interleaved PCM read as container values."""
    import bench
    import torch
    wls = bench.build_library(0, bench.host_cores())
    files = []
    for wl in wls:
        packets = [bytes(wl['packed'][int(o):int(o) + int(z)]) for o, z in zip(wl['offsets'], wl['sizes'])]
        files.append(build_m4a(wl['cookie'], packets, bits=wl['bits'], last_frames=wl['frames'] % 4096)[0])
    libd = pkg.NewLibraryDecoder((0,))
    try:
        res = libd.DecodeTracks([pkg.Track(wl['cookie'], wl['packed'], wl['offsets'], wl['sizes']) for wl in wls])
    finally:
        libd.close()
    want = []
    for wl, r in zip(wls, res):
        assert r.err is None and (r.status == 0).all()
        nbytes = int(r.out_bytes.sum())
        assert r.pcm.shape[1] == r.out_bytes[0]  # full packets back to back: the PCM is contiguous
        raw = torch.from_numpy(r.pcm.reshape(-1)[:nbytes]).cuda()
        if wl['bits'] == 16:
            v = raw.view(torch.int16).int()
        else:
            b = raw.view(-1, 3).int()
            v = b[:, 0] | (b[:, 1] << 8) | (b[:, 2].to(torch.uint8).view(torch.int8).int() << 16)
        want.append(v.view(-1, 2).t())
    for dtype in (torch.float32, torch.int32):
        got = pkg.LoadTracks(files, 0, dtype)
        for wl, g, w in zip(wls, got, want):
            assert g.err is None and g.format == pkg.PCMFormat(44100, wl['bits'], 2)
            assert g.samples.shape == (2, wl['frames']) and g.samples.dtype == dtype
            expect = w if dtype == torch.int32 else w.float() * 2.0 ** -(15 if wl['bits'] == 16 else 23)
            assert torch.equal(g.samples, expect), wl['name']
        del got
