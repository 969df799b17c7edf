#!/usr/bin/env python
"""tools/planar_bench.py -- what channel-planar output on the device costs (one JSON line on stdout).

    python tools/planar_bench.py [--steps N] [--warmup W] [--workloads c1,c2,c3,c4] [--device D]

Per workload (bench.py's streams and seeds, packets resident in HBM), on one GPU in one process, the arms alternate
step by step and each call is timed with CUDA events on one stream:

  interleaved   alacb200_decode_packets_device into slots of frame_bytes rounded up to 16 (the layout of the planar
                path's intermediate, so the decode kernel does the same work in both arms)
  s32 / f32     alacb200_decode_planar_device (s16 too on the 16-bit c1): decode + frame scan + planar pass
  pass_ms       median over steps of (planar - interleaved) of the same step: the scan, the planar pass and the
                stream-ordered allocation of the intermediate
  pass_gbs      (PCM bytes read from the intermediate + sample bytes written) / pass_ms, against MEASURED_PEAKS.json hbm_gbs

LoadTrack on the 60 s c1 M4A against what a caller does without it: NewDecoder(...).ReadAll(), unpacking the PCM into
channel-planar samples and uploading them (host clock, median over alternating repetitions, each ending in a device
synchronisation). The line carries the GPU's name, power limit and max SM clock, queried in the same run.

`tracks`: many files in one call, for two batches of M4A images (bench.py's encoder, tests/m4a_writer.build_m4a):
  lib     bench.build_library(0, ...): 32 tracks of 3 min of 44.1 kHz stereo, 16- and 24-bit alternating
  clips   256 clips of 10 s of 44.1 kHz stereo, 16- and 24-bit alternating (the dataset regime)
Per batch, arms alternating: LoadTracks against a loop of LoadTrack (host clock up to a device synchronise, float32);
LibraryDecoder.DecodePlanar over the whole device-resident batch (ordered by config) against a loop of per-track
PacketDecoder.DecodePlanar (one decoder per config; CUDA events on one stream); and, in a separate profiled run,
the alac_decode_kernel* launches of one call of each.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

import bench  # noqa: E402 -- build_workload, its stream cache and the measured peak

SEEDS = {'c1': 1, 'c2': 2, 'c3': 2, 'c4': 4}  # the seeds bench.py decodes each workload with


def gpu_info(dev):
    q = 'name,power.limit,clocks.max.sm'
    try:
        out = subprocess.run(['nvidia-smi', '-i', str(dev), f'--query-gpu={q}', '--format=csv,noheader,nounits'],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, mhz = [f.strip() for f in out.split(',')]
        return {'name': name, 'power_limit_w': float(power), 'max_sm_mhz': float(mhz)}
    except Exception as e:  # noqa: BLE001 -- the line says what is missing instead of failing the run
        return {'error': f'nvidia-smi query failed: {e}'}


def time_arms(torch, stream, arms, steps, warmup):
    """arms: {name: callable enqueuing one call on `stream`} -> {name: [ms per step]}, arms alternating."""
    for f in arms.values():
        for _ in range(warmup):
            f()
    torch.cuda.synchronize()
    ev = {k: [] for k in arms}
    for _ in range(steps):
        for k, f in arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            f()
            e1.record(stream)
            ev[k].append((e0, e1))
    torch.cuda.synchronize()
    return {k: [a.elapsed_time(b) for a, b in v] for k, v in ev.items()}


def planar_workload(pkg, torch, dev, wl, steps, warmup, peak):
    n = len(wl['sizes'])
    ch, bits = wl['channels'], wl['bits']
    bps = pkg.BytesPerSample(bits)
    dec = pkg.NewPacketDecoder(pkg.ParseMagicCookie(wl['cookie']), dev)
    fl = wl['cfg'].frame_length
    slot = (dec.frame_bytes + 15) // 16 * 16
    d_packed = torch.from_numpy(np.ascontiguousarray(wl['packed'])).to(dev)
    d_off = torch.from_numpy(wl['offsets'].view(np.int64)).to(dev)
    d_sz = torch.from_numpy(wl['sizes'].view(np.int32)).to(dev)
    d_pcm = torch.empty(n * slot, dtype=torch.uint8, device=dev)
    d_nb = torch.empty(n, dtype=torch.int32, device=dev)
    d_st = torch.empty(n, dtype=torch.int32, device=dev)
    types = {'s32': (pkg.SAMPLES_S32, torch.int32), 'f32': (pkg.SAMPLES_F32, torch.float32)}
    if bits == 16:
        types['s16'] = (pkg.SAMPLES_S16, torch.int16)
    outs = {k: torch.empty((ch, n * fl), dtype=t, device=dev) for k, (_, t) in types.items()}
    d_fs = torch.empty(n + 1, dtype=torch.int64, device=dev)
    stream = torch.cuda.Stream(dev)

    def check(rc, what):
        if rc != 0:
            raise RuntimeError(f'{what} rc={rc}: {pkg.lib.alacb200_last_error().decode()}')

    def interleaved():
        check(pkg.lib.alacb200_decode_packets_device(dec._h, d_packed.data_ptr(), d_packed.numel(), d_off.data_ptr(), d_sz.data_ptr(), n,
                                                     d_pcm.data_ptr(), slot, d_nb.data_ptr(), d_st.data_ptr(), stream.cuda_stream),
              'alacb200_decode_packets_device')

    def planar(k):
        st, out = types[k][0], outs[k]
        return lambda: check(pkg.lib.alacb200_decode_planar_device(dec._h, d_packed.data_ptr(), d_packed.numel(), d_off.data_ptr(),
                                                                   d_sz.data_ptr(), n, st, out.data_ptr(), n * fl, d_fs.data_ptr(),
                                                                   d_st.data_ptr(), stream.cuda_stream), 'alacb200_decode_planar_device')

    arms = {'interleaved': interleaved}
    arms.update({k: planar(k) for k in types})
    # gate: every packet decodes, the totals add up, and the S32 samples of the first 64 packets are the interleaved PCM
    for f in arms.values():
        f()
    torch.cuda.synchronize()
    assert int((d_st != 0).sum()) == 0 and int(d_fs[n]) == wl['frames'], 'decode errors or a wrong total'
    k = min(n, 64)
    rows = d_pcm.view(n, slot)[:k, :dec.frame_bytes].cpu().numpy()
    nb = d_nb[:k].cpu().numpy()
    import oracle_lib as ol
    want = np.concatenate([ol.pcm_bytes_to_int(rows[i, :nb[i]].tobytes(), bits, ch) for i in range(k)]).T
    f_k = int(d_fs[k])
    assert np.array_equal(outs['s32'][:, :f_k].cpu().numpy(), want.astype(np.int32)), 'planar S32 differs from the interleaved PCM'
    ms = time_arms(torch, stream, arms, steps, warmup)
    base = ms['interleaved']
    samples = wl['frames'] * ch
    rec = {'packets': n, 'frames': wl['frames'], 'channels': ch, 'bits': bits, 'interleaved_ms': float(np.mean(base)), 'planar': {}}
    for k, (_, t) in types.items():
        diff = float(np.median(np.subtract(ms[k], base)))
        read, written = samples * bps, samples * torch.empty((), dtype=t).element_size()
        gbs = (read + written) / (diff / 1e3) / 1e9 if diff > 0 else None
        rec['planar'][k] = {'ms': float(np.mean(ms[k])), 'pass_ms': diff, 'pass_bytes_read': read, 'pass_bytes_written': written,
                            'pass_gbs': gbs, 'pass_frac_of_peak': gbs / peak if gbs else None,
                            'over_interleaved': float(np.mean(ms[k]) / np.mean(base))}
    dec.close()
    del d_pcm, outs
    torch.cuda.empty_cache()
    return rec


def load_track_leg(pkg, torch, dev, reps):
    """LoadTrack vs NewDecoder + ReadAll + unpack + upload on the c1 M4A, for float32 and int16."""
    from m4a_writer import build_m4a
    wl = bench.build_workload('c1', seed=SEEDS['c1'], threads=bench.host_cores())
    packets = [bytes(wl['packed'][int(o):int(o) + int(z)]) for o, z in zip(wl['offsets'], wl['sizes'])]
    data, _ = build_m4a(wl['cookie'], packets, last_frames=wl['frames'] % 4096)

    def today(dtype):
        d = pkg.NewDecoder(data, dev)
        pcm = d.ReadAll()
        d.close()
        x = torch.from_numpy(np.frombuffer(pcm, dtype=np.int16).reshape(-1, 2)).to(dev)
        out = x.t().float() * 2.0 ** -15 if dtype == torch.float32 else x.t().contiguous()
        torch.cuda.synchronize(dev)
        return out

    def new(dtype):
        out, _ = pkg.LoadTrack(data, dev, dtype)
        torch.cuda.synchronize(dev)
        return out

    rec = {'file_bytes': len(data), 'frames': wl['frames'], 'reps': reps}
    for name, dtype in (('f32', torch.float32), ('s16', torch.int16)):
        assert torch.equal(today(dtype), new(dtype)), 'LoadTrack differs from ReadAll'
        t = {'load_track': [], 'read_all_unpack_upload': []}
        for _ in range(reps):
            for k, f in (('load_track', new), ('read_all_unpack_upload', today)):
                t0 = time.perf_counter()
                f(dtype)
                t[k].append((time.perf_counter() - t0) * 1e3)
        rec[name] = {k + '_ms': float(np.median(v)) for k, v in t.items()}
    return rec


def tracks_leg(pkg, torch, dev, reps, steps, warmup):
    from m4a_writer import build_m4a
    from torch.profiler import ProfilerActivity, profile
    threads = bench.host_cores()
    batches = {'lib': [(wl['bits'], wl['cookie'], wl['packed'], wl['offsets'], wl['sizes'], wl['frames'])
                       for wl in bench.build_library(0, threads)]}
    import oracle_lib as ol
    clips = []
    for k in range(256):
        bits = 16 if k % 2 == 0 else 24
        packed, offs, sizes = bench.encode_track(bits, 2, 44100, 441000, seed=5000 + k, threads=threads, tag='clip')
        clips.append((bits, ol.make_cookie(ol.Config.make(bit_depth=bits, num_channels=2, sample_rate=44100)), packed, offs, sizes, 441000))
    batches['clips'] = clips
    rec = {}
    for name, tracks in batches.items():
        files = []
        for bits, cookie, packed, offs, sizes, frames in tracks:
            packets = [bytes(packed[int(o):int(o) + int(z)]) for o, z in zip(offs, sizes)]
            files.append(build_m4a(cookie, packets, bits=bits, last_frames=frames % 4096)[0])
        # 1. LoadTracks vs a loop of LoadTrack
        def one_call():
            out = pkg.LoadTracks(files, dev)
            torch.cuda.synchronize(dev)
            return out

        def loop():
            out = [pkg.LoadTrack(f, dev) for f in files]
            torch.cuda.synchronize(dev)
            return out
        a, b = one_call(), loop()
        assert all(x.err is None and torch.equal(x.samples, y[0]) for x, y in zip(a, b)), 'LoadTracks differs from LoadTrack'
        del a, b
        t = {'load_tracks': [], 'load_track_loop': []}
        for _ in range(reps):
            for k, f in (('load_tracks', one_call), ('load_track_loop', loop)):
                t0 = time.perf_counter()
                f()
                t[k].append((time.perf_counter() - t0) * 1e3)
        r = {'tracks': len(files), 'packets': int(sum(len(x[4]) for x in tracks)), 'frames': int(sum(x[5] for x in tracks)),
             'file_bytes': int(sum(len(f) for f in files)), 'reps': reps}
        r.update({k + '_ms': float(np.median(v)) for k, v in t.items()})
        # 2. device-resident: one library call vs per-track PacketDecoder.DecodePlanar, batch ordered by config
        order = sorted(range(len(tracks)), key=lambda i: tracks[i][0])
        parts, offs_all, sizes_all, base = [], [], [], 0
        for i in order:
            packed, offs, sizes = tracks[i][2], tracks[i][3], tracks[i][4]
            span = (len(packed) + 15) // 16 * 16
            parts.append(np.pad(packed, (0, span - len(packed))))
            offs_all.append(offs.astype(np.int64) + base)
            sizes_all.append(sizes.view(np.int32))
            base += span
        d_packed = torch.from_numpy(np.concatenate(parts)).to(dev)
        d_off = torch.from_numpy(np.concatenate(offs_all)).to(dev)
        d_sz = torch.from_numpy(np.concatenate(sizes_all)).to(dev)
        counts = [len(tracks[i][4]) for i in order]
        starts = np.concatenate([[0], np.cumsum(counts)])
        cookies = [tracks[i][1] for i in order]
        libd = pkg.NewLibraryDecoder((dev,))
        decs = {c: pkg.NewPacketDecoder(pkg.ParseMagicCookie(c), dev) for c in set(cookies)}
        stream = torch.cuda.Stream(dev)
        keep = []

        def lib_call():
            with torch.cuda.stream(stream):
                keep.append(libd.DecodePlanar(d_packed, d_off, d_sz, cookies, counts, device=dev))

        def per_track():
            with torch.cuda.stream(stream):
                for k, c in enumerate(cookies):
                    a, b = int(starts[k]), int(starts[k + 1])
                    keep.append(decs[c].DecodePlanar(d_packed, d_off[a:b], d_sz[a:b]))

        def drop(f):
            def g():
                f()
                keep.clear()  # the caching allocator reuses the outputs on the same stream
            return g
        ms = time_arms(torch, stream, {'library_decode_planar': drop(lib_call), 'per_track_decode_planar': drop(per_track)}, steps, warmup)
        r.update({k + '_ms': float(np.median(v)) for k, v in ms.items()})
        # 3. decode launches per call, in a separate profiled run
        def launches(f):
            torch.cuda.synchronize(dev)
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                f()
                torch.cuda.synchronize(dev)
            return sum('alac_decode_kernel' in e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA)
        r['decode_launches'] = {'load_tracks': launches(one_call), 'load_track_loop': launches(loop),
                                'library_decode_planar': launches(drop(lib_call)), 'per_track_decode_planar': launches(drop(per_track))}
        for d in decs.values():
            d.close()
        libd.close()
        del d_packed, d_off, d_sz
        torch.cuda.empty_cache()
        rec[name] = r
    return rec


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--reps', type=int, default=20, help='repetitions of each LoadTrack arm')
    ap.add_argument('--workloads', default='c1,c2,c3,c4')
    ap.add_argument('--device', type=int, default=0)
    ap.add_argument('--tracks-only', action='store_true', help='only the `tracks` record')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be >= 1')
    import torch
    from alac_b200_loader import load_package
    pkg = load_package()
    if not torch.cuda.is_available() or pkg.lib.alacb200_device_count() < 1:
        raise SystemExit('planar_bench.py needs a CUDA device')
    dev = args.device
    torch.cuda.set_device(dev)
    peak, peak_src = bench.measured_peak_gbs()
    line = {'tool': 'tools/planar_bench.py', 'gpu': gpu_info(dev), 'steps': args.steps, 'warmup': args.warmup,
            'peak_gbs': peak, 'peak_source': peak_src, 'workloads': {}}
    if not args.tracks_only:
        for name in args.workloads.split(','):
            wl = bench.build_workload(name, seed=SEEDS[name], threads=bench.host_cores())
            line['workloads'][name] = planar_workload(pkg, torch, dev, wl, args.steps, args.warmup, peak)
        line['load_track'] = load_track_leg(pkg, torch, dev, args.reps)
    line['tracks'] = tracks_leg(pkg, torch, dev, args.reps, args.steps, args.warmup)
    print(json.dumps(line))


if __name__ == '__main__':
    main()
