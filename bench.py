#!/usr/bin/env python
"""bench.py -- throughput of the ALAC packet-decode hot path on B200 (one JSON line on stdout).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c3] [--only-main]
                    [--dump-outputs DIR]

A "step" is one pass of the hot path over the whole batch. The headline workload is BASELINE configs[2] -- the largest
config that fits one GPU: 24-bit stereo 192 kHz with bytesShifted=1, 1 h, 168 750 packets of 4096 frames. With --gpus N
(one rank per GPU under torchrun) that ONE batch is cut by the product's own partitioner (shard_ranges: contiguous
packet ranges balanced by compressed bytes, no data-path collective) -- strong scaling; every rank times its shard and
the line reports the max over ranks.

  value       whole-job decoded channel-samples/s with packets resident in HBM (CUDA events on the launch stream)
  e2e         same through the host C-ABI call (alacb200_decode_packets) with pinned HOST buffers: H2D of the
              compressed bytes and D2H of the PCM are inside the timed region
  roofline    decode kernel: (compressed bytes in + PCM bytes out) / its event-timed duration vs the measured HBM peak
  cpu_baseline / --impl reference   the CPU oracle (C restatement of the Go reference; no Go toolchain in this image) on
              all host cores, same packets
  workloads   (N=1) the other BASELINE configs as sub-records -- c1, c2, c4 and `lib`, a configs[4]-style library of mixed
              16/24-bit tracks through the multi-track entry point -- each with value, e2e, roofline fraction and a bounded
              CPU sample; plus c2 re-encoded by FFmpeg's encoder (encoder realism check)
  lib_weak    (every N) the library batch with one track list PER RANK: weak scaling of the multi-track path
  e2e_api     (N=1) what a caller of the drop-in API pays, through the compiled C++ mirror of the Go package:
              PacketDecoder::DecodePackets over all of c2, NewDecoder + Read over the c1 M4A

Streams come from the test-side encoder on the seeded SURVEY.md section 8d signal (cached in a per-user temporary
directory, $ALAC_B200_CACHE to override). The in-run gate checks 64 packets per workload against the oracle before timing;
the full-size bit-exact checks live in tests/.

--dump-outputs DIR writes what the timed path of the headline workload returned in its last step, so that two builds can
be compared output for output (the inputs are the same seeded streams from run to run):
  pcm.npy          float32 [k, frame_length, channels] decoded samples of a fixed seeded sample of k packets (float64 for
                   32-bit streams; samples past a packet's out_bytes are 0), at most ~56 MB
  pcm_packets.npy  float64 [k] the indices of those packets in the batch (the first and the short last one included)
  out_bytes.npy    float64 [n] PCM bytes of every packet
  status.npy       float64 [n] status word of every packet
With --gpus N the shards are gathered on rank 0, so the files do not depend on N; --impl reference writes the same files
from the CPU oracle.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

SIGNALS = {'lsb': 'lsb'}  # workload -> signal kind (default 'bench')
WORKLOADS = {
    # name: (bits, channels, rate, seconds, description)
    'c1': (16, 2, 44100, 60, '16-bit stereo 44.1 kHz, 60 s (BASELINE configs[0])'),
    'c2': (24, 2, 96000, 600, '24-bit stereo 96 kHz, 10 min, batched DecodePackets (BASELINE configs[1])'),
    'c3': (24, 2, 192000, 3600, '24-bit stereo 192 kHz with shift buffer (bytesShifted=1), 1 h (BASELINE configs[2])'),
    'c4': (24, 8, 48000, 1800, '7.1 24-bit 48 kHz, 30 min (BASELINE configs[3])'),
    'c3q': (24, 2, 192000, 900, '24-bit stereo 192 kHz with shift buffer, 15 min: the shard one of four GPUs gets of c3 (developer: wave quantisation)'),
    'lib16': (16, 2, 44100, 48 * 180, '48 x 3 min of 16-bit stereo 44.1 kHz in one call, 93 k packets (throughput regime, one depth)'),
    'lsb': (24, 2, 96000, 120, '24-bit stereo 96 kHz, 2 min of +-2 LSB noise: the quiet-passage regime only (developer stress)'),
    'smoke': (24, 2, 96000, 20, '24-bit stereo 96 kHz, 20 s (quick self-test)'),
}
LIB_TRACKS = 32  # tracks per rank of the library batch: half 16-bit, half 24-bit, 3 min of 44.1 kHz stereo each (configs[4])
LIB_DESC = ('library batch (BASELINE configs[4] scaled to one call per GPU): %d distinct stereo 44.1 kHz tracks of 3 min, half 16-bit '
            'half 24-bit, decoded through alacb200_library_decode_tracks' % LIB_TRACKS)


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def _cache_dir():
    # per user: a cache directory another user created first would not be writable
    d = os.environ.get('ALAC_B200_CACHE') or os.path.join(tempfile.gettempdir(), f'alac_b200_cache_{os.getuid()}')
    os.makedirs(d, exist_ok=True)
    return d


def encode_track(bits, ch, rate, frames, seed, threads, kind='bench', tag=None):
    """-> (packed u8, offsets u64, sizes u32) of one track from the test-side encoder; cached in _cache_dir()."""
    import oracle_lib as ol
    from signals import make_signal
    path = os.path.join(_cache_dir(), f'{tag or "t"}_{bits}_{ch}_{rate}_{frames}_{kind}_seed{seed}_v1.npz')
    if os.path.exists(path):
        z = np.load(path)
        return z['packed'], z['offsets'], z['sizes']
    cfg = ol.Config.make(bit_depth=bits, num_channels=ch, sample_rate=rate)
    fl = cfg.frame_length
    npk = (frames + fl - 1) // fl
    seg = 256  # packets per work item
    items = [(a, min(npk, a + seg)) for a in range(0, npk, seg)]
    results = [None] * len(items)

    def work(k):
        a, b = items[k]
        f0, f1 = a * fl, min(frames, b * fl)
        x = make_signal(kind, ch, f1 - f0, bits, rate, seed=seed * 100003 + k, t0=f0)
        results[k] = ol.encode_stream(cfg, x)

    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(max_workers=max(1, threads)) as ex:
        list(ex.map(work, range(len(items))))
    packed, offsets, sizes = ol.pack([p for r in results for p in r])
    tmp = path + f'.{os.getpid()}.tmp.npz'
    np.savez(tmp, packed=packed, offsets=offsets, sizes=sizes)
    os.replace(tmp, path)
    return packed, offsets, sizes


def build_workload(name, seed, threads):
    """-> dict(cfg, cookie, packed u8, offsets u64, sizes u32, frames, channels, bits, rate). Cached in _cache_dir()."""
    import oracle_lib as ol
    bits, ch, rate, seconds, _ = WORKLOADS[name]
    cfg = ol.Config.make(bit_depth=bits, num_channels=ch, sample_rate=rate)
    frames = rate * seconds
    packed, offsets, sizes = encode_track(bits, ch, rate, frames, seed, threads, SIGNALS.get(name, 'bench'), tag=name)
    return dict(name=name, cfg=cfg, cookie=ol.make_cookie(cfg), packed=packed, offsets=offsets, sizes=sizes, frames=frames,
                channels=ch, bits=bits, rate=rate, seconds=seconds)


def build_ffmpeg_workload(seconds=600):
    """configs[1]'s shape encoded by FFmpeg's ALAC encoder (the reference's own conformance encoder) instead of the
    test-side one. -> workload dict, or None when the FFmpeg libraries are not importable."""
    import oracle_lib as ol
    from signals import make_signal
    sys.path.insert(0, os.path.join(ROOT, 'tests', 'golden'))
    path = os.path.join(_cache_dir(), f'c2_ffmpeg_{seconds}_v1.npz')
    bits, ch, rate = 24, 2, 96000
    frames = rate * seconds
    if os.path.exists(path):
        z = np.load(path)
        packed, offsets, sizes, cookie = z['packed'], z['offsets'], z['sizes'], bytes(z['cookie'])
    else:
        try:
            import ffmpeg_alac as ff
        except Exception:
            return None
        x = make_signal('bench', ch, frames, bits, rate, seed=2)
        cookie, packets = ff.alac_encode(np.ascontiguousarray(x.T), bits, rate, {})
        packed, offsets, sizes = ol.pack(packets)
        tmp = path + f'.{os.getpid()}.tmp.npz'
        np.savez(tmp, packed=packed, offsets=offsets, sizes=sizes, cookie=np.frombuffer(cookie, dtype=np.uint8))
        os.replace(tmp, path)
    st, cfg = ol.parse_cookie(cookie)
    assert st == 0
    return dict(name='c2_ffmpeg', cfg=cfg, cookie=cookie, packed=packed, offsets=offsets, sizes=sizes, frames=frames, channels=ch,
                bits=bits, rate=rate, seconds=seconds)


def build_library(rank, threads):
    """-> list of workload dicts, one per track: LIB_TRACKS distinct tracks per rank, 16- and 24-bit alternating."""
    import oracle_lib as ol
    tracks = []
    for t in range(LIB_TRACKS):
        bits = 16 if t % 2 == 0 else 24
        cfg = ol.Config.make(bit_depth=bits, num_channels=2, sample_rate=44100)
        frames = 44100 * 180
        packed, offsets, sizes = encode_track(bits, 2, 44100, frames, seed=1000 + rank * LIB_TRACKS + t, threads=threads, tag='lib')
        tracks.append(dict(name=f'lib{t}', cfg=cfg, cookie=ol.make_cookie(cfg), packed=packed, offsets=offsets, sizes=sizes,
                           frames=frames, channels=2, bits=bits, rate=44100, seconds=180))
    return tracks


def bind_to_gpu_numa(dev):
    """Pin this rank's threads to the NUMA node of its GPU before any pinned buffer is allocated (first touch), so the
    H2D / D2H copies of the end-to-end leg do not cross sockets when several ranks run at once. Best effort."""
    try:
        out = subprocess.run(['nvidia-smi', '-i', str(dev), '--query-gpu=pci.bus_id', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        bus = out[-12:] if len(out) >= 12 else out  # 00000000:1B:00.0 -> 0000:1b:00.0
        node = int(open(f'/sys/bus/pci/devices/{bus}/numa_node').read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f'/sys/devices/system/node/node{node}/cpulist').read().strip().split(','):
            a, _, b = part.partition('-')
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:
        pass
    return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, dev):
        self.dev, self.proc, self.lines = dev, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.dev), f'--query-gpu={self.Q}',
                                          '--format=csv,noheader,nounits', '-lms', '100'], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for ln in self.lines:
            f = [x.strip() for x in ln.split(',')]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(nm)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm)}


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            return float(json.load(f)['hbm_gbs']), 'MEASURED_PEAKS.json hbm_gbs (of measured)'
    except Exception:
        return 6650.0, 'B200_PROFILING.md fallback 6.65 TB/s (of fallback)'


def run_cpu(wl, threads, min_seconds, max_rounds=50, max_packets=None):
    """Oracle on `threads` host threads over (a prefix of) the workload, repeated until min_seconds.
    -> (samples/s, rounds, seconds, packets per round)"""
    import oracle_lib as ol
    n = len(wl['sizes']) if max_packets is None else min(len(wl['sizes']), max_packets)
    offs, sizes = wl['offsets'][:n], wl['sizes'][:n]
    out = np.zeros((n, wl['cfg'].frame_bytes()), dtype=np.uint8)
    out[:] = 1  # touch the pages outside the timed region
    _, nb, _ = ol.decode_batch(wl['cfg'], wl['packed'], offs, sizes, nthreads=threads, out=out)  # warm-up
    samples = int(nb.astype(np.int64).sum()) // wl['cfg'].bps()
    rounds, t0 = 0, time.perf_counter()
    while True:
        _, _, st = ol.decode_batch(wl['cfg'], wl['packed'], offs, sizes, nthreads=threads, out=out)
        rounds += 1
        dt = time.perf_counter() - t0
        if dt >= min_seconds or rounds >= max_rounds:
            break
    assert (st == 0).all()
    return samples * rounds / dt, rounds, dt, n


def emit_line(line):
    """The ONE JSON line of the contract, written to the real stdout (see main)."""
    os.write(_REAL_STDOUT, (json.dumps(line) + '\n').encode())


_REAL_STDOUT = 1

DUMP_BYTES = 56 << 20  # everything --dump-outputs writes stays under 64 MB


def dump_dtype(bits):
    return np.float32 if bits <= 24 else np.float64  # float32 holds every 24-bit sample exactly


def dump_index(n, wl):
    """The packets whose PCM --dump-outputs writes: a fixed seeded sample of the batch's n packets that fits DUMP_BYTES
    next to the per-packet arrays, plus the first packet and the last (the short one)."""
    per_packet = wl['cfg'].frame_length * wl['channels'] * np.dtype(dump_dtype(wl['bits'])).itemsize + 8
    k = min(n, max(1, (DUMP_BYTES - 16 * n) // per_packet))
    idx = np.random.default_rng(0).choice(n, size=k, replace=False)
    return np.union1d(idx, [0, n - 1]).astype(np.int64)


def write_dump(path, wl, idx, rows, out_bytes, status):
    """rows: u8 [len(idx), >= frame_bytes], the PCM the timed path returned for packets idx; out_bytes, status: [n] of
    every packet. Writes the arrays described in the module docstring."""
    import oracle_lib as ol
    ch, fl, bps = wl['channels'], wl['cfg'].frame_length, wl['cfg'].bps()
    rows = np.ascontiguousarray(rows[:, :fl * ch * bps])
    pcm = ol.pcm_bytes_to_int(rows.tobytes(), wl['bits'], ch).reshape(len(idx), fl * ch)
    valid = np.where(status[idx] == 0, out_bytes[idx], 0).astype(np.int64) // bps
    pcm[np.arange(fl * ch)[None, :] >= valid[:, None]] = 0  # bytes past out_bytes are not part of the result
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, 'pcm.npy'), pcm.reshape(len(idx), fl, ch).astype(dump_dtype(wl['bits'])))
    np.save(os.path.join(path, 'pcm_packets.npy'), idx.astype(np.float64))
    np.save(os.path.join(path, 'out_bytes.npy'), np.asarray(out_bytes).astype(np.float64))
    np.save(os.path.join(path, 'status.npy'), np.asarray(status).astype(np.float64))


class Pinned:
    """A pinned host array from the product's allocator."""

    def __init__(self, pkg, nbytes):
        self.pkg, self.nbytes = pkg, max(1, int(nbytes))
        self.ptr = pkg.lib.alacb200_pinned_alloc(self.nbytes)
        if not self.ptr:
            raise MemoryError('alacb200_pinned_alloc failed')
        self.arr = np.ctypeslib.as_array(C.cast(self.ptr, C.POINTER(C.c_uint8)), shape=(self.nbytes,))

    def free(self):
        if self.ptr:
            self.pkg.lib.alacb200_pinned_free(self.ptr)
            self.ptr = None


class Runner:
    """One workload (or one rank's shard of it) on one device: the device-resident leg, the host C-ABI leg, the gate."""

    def __init__(self, pkg, torch, dev, wl, lo=0, hi=None):
        self.pkg, self.torch, self.wl = pkg, torch, wl
        hi = len(wl['sizes']) if hi is None else hi
        self.n = hi - lo
        self.offsets = np.ascontiguousarray(wl['offsets'][lo:hi])
        self.sizes = np.ascontiguousarray(wl['sizes'][lo:hi])
        self.comp_bytes = int(self.sizes.astype(np.int64).sum())
        self.dec = pkg.NewPacketDecoder(pkg.ParseMagicCookie(wl['cookie']), dev)
        self.bps = pkg.BytesPerSample(wl['bits'])
        self.stride = (self.dec.frame_bytes + 15) // 16 * 16
        fl = wl['cfg'].frame_length
        self.frames = min(wl['frames'], hi * fl) - lo * fl  # frames of this shard (the last packet of the track may be short)
        self.samples = self.frames * wl['channels']
        self.pcm_bytes = self.samples * self.bps
        self.stream = torch.cuda.Stream()
        # device-resident buffers (torch is plumbing: memory + streams + events). The shard's bytes only.
        if self.n:
            b0 = int(self.offsets[0]) & ~15
            b1 = int(self.offsets[-1]) + int(self.sizes[-1])
        else:
            b0 = b1 = 0
        self.host_bytes = wl['packed'][b0:b1 + 64] if b1 + 64 <= len(wl['packed']) else np.concatenate([wl['packed'][b0:], np.zeros(64, np.uint8)])
        self.rel_offsets = (self.offsets - np.uint64(b0)).astype(np.uint64)
        self.d_packed = torch.from_numpy(np.ascontiguousarray(self.host_bytes)).cuda()
        self.d_offsets = torch.from_numpy(self.rel_offsets.view(np.int64)).cuda()
        self.d_sizes = torch.from_numpy(self.sizes.view(np.int32)).cuda()
        self.d_pcm = torch.empty(max(1, self.n) * self.stride, dtype=torch.uint8, device='cuda')
        self.d_nb = torch.zeros(max(1, self.n), dtype=torch.int32, device='cuda')
        self.d_st = torch.zeros(max(1, self.n), dtype=torch.int32, device='cuda')
        self.h_in = self.h_out = None

    def step_device(self):
        rc = self.pkg.lib.alacb200_decode_packets_device(self.dec._h, self.d_packed.data_ptr(), self.d_packed.numel(), self.d_offsets.data_ptr(),
                                                         self.d_sizes.data_ptr(), self.n, self.d_pcm.data_ptr(), self.stride, self.d_nb.data_ptr(),
                                                         self.d_st.data_ptr(), self.stream.cuda_stream)
        if rc != 0:
            raise RuntimeError(f'decode_packets_device rc={rc}: {self.pkg.lib.alacb200_last_error().decode()}')

    def gate(self, cores):
        """Before timing: all packets OK, the PCM of a sample of packets equals the oracle's."""
        import oracle_lib as ol
        self.step_device()
        self.torch.cuda.synchronize()
        assert int((self.d_st[:self.n] != 0).sum().item()) == 0, 'decode errors in the bench workload'
        k = min(self.n, 64)
        self.want, _, _ = ol.decode_batch(self.wl['cfg'], self.wl['packed'], self.offsets[:k], self.sizes[:k], nthreads=min(cores, 8))
        got = self.d_pcm.view(max(1, self.n), self.stride)[:k, :self.dec.frame_bytes].cpu().numpy()
        assert np.array_equal(got, self.want), 'GPU PCM differs from the oracle'
        return k

    def time_device(self, steps, warmup, barrier):
        torch = self.torch
        for _ in range(warmup):
            self.step_device()
        barrier()
        self.dec.set_profiling(True)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(self.stream):
            e0.record(self.stream)
            for _ in range(steps):
                self.step_device()
            e1.record(self.stream)
        barrier()
        prof = self.dec.get_profile()
        self.dec.set_profiling(False)
        return e0.elapsed_time(e1), prof.ms_decode / max(1, prof.launches_decode), int(prof.launches_decode)

    def device_results(self, idx):
        """What the last device step returned: (PCM rows of this shard's packets idx, out_bytes and status of all)."""
        torch = self.torch
        torch.cuda.synchronize()
        sel = torch.from_numpy(np.ascontiguousarray(idx, dtype=np.int64)).cuda()
        rows = self.d_pcm.view(max(1, self.n), self.stride)[sel, :self.dec.frame_bytes].cpu().numpy()
        return rows, self.d_nb[:self.n].cpu().numpy().view(np.uint32), self.d_st[:self.n].cpu().numpy()

    def prepare_host(self):
        self.h_in = Pinned(self.pkg, len(self.host_bytes))
        self.h_in.arr[:len(self.host_bytes)] = self.host_bytes
        self.h_out = Pinned(self.pkg, max(1, self.n) * self.stride)
        self.h_out.arr[:] = 0
        self.h_nb = np.zeros(max(1, self.n), dtype=np.uint32)
        self.h_st = np.zeros(max(1, self.n), dtype=np.int32)

    def step_host(self):
        rc = self.pkg.lib.alacb200_decode_packets(self.dec._h, self.h_in.ptr, len(self.host_bytes), self.rel_offsets.ctypes.data, self.sizes.ctypes.data,
                                                  self.n, self.h_out.ptr, self.stride, self.h_nb.ctypes.data, self.h_st.ctypes.data)
        if rc != 0:
            raise RuntimeError(f'decode_packets rc={rc}: {self.pkg.lib.alacb200_last_error().decode()}')

    def time_host(self, steps, barrier):
        self.prepare_host()
        for _ in range(2):
            self.step_host()
        k = len(self.want)
        assert (self.h_st[:self.n] == 0).all() and np.array_equal(self.h_out.arr[:self.n * self.stride].reshape(self.n, self.stride)[:k, :self.dec.frame_bytes], self.want)
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            self.step_host()
        self.torch.cuda.synchronize()
        return time.perf_counter() - t0

    def bytes_per_step(self):
        return self.comp_bytes + 12 * self.n, max(0, self.n - 1) * self.stride + self.dec.frame_bytes + 8 * self.n

    def close(self):
        for p in (self.h_in, self.h_out):
            if p:
                p.free()
        self.dec.close()
        del self.d_packed, self.d_pcm


def sub_record(pkg, torch, dev, wl, cores, steps, peak, cpu_seconds=2.5, with_cpu=True):
    """value / e2e / roofline fraction / bounded CPU sample of one more workload on one GPU."""
    r = Runner(pkg, torch, dev, wl)
    gate = r.gate(cores)
    sync = torch.cuda.synchronize
    ms_total, dec_ms, launches = r.time_device(steps, 3, sync)
    e2e_steps = max(3, min(steps, 6))
    e2e_s = r.time_host(e2e_steps, sync)
    algo = r.comp_bytes + r.pcm_bytes
    rec = {'workload': f"{wl['name']}: {WORKLOADS.get(wl['name'], (0, 0, 0, 0, 'configs[1] shape, FFmpeg-encoded'))[4]}", 'packets': r.n,
           'value': r.samples * steps / (ms_total / 1e3), 'unit': 'samples/s', 'ms_per_step': ms_total / steps,
           'x_realtime': r.samples * steps / (ms_total / 1e3) / wl['channels'] / wl['rate'],
           'e2e': {'value': r.samples * e2e_steps / e2e_s, 'ms_per_step': e2e_s / e2e_steps * 1e3},
           'roofline_frac': algo / (dec_ms / 1e3) / 1e9 / peak, 'kernel_ms': dec_ms, 'gpu_launches_per_step': launches // max(1, steps),
           'compressed_bytes': r.comp_bytes, 'pcm_bytes': r.pcm_bytes, 'gate_packets_vs_oracle': gate}
    if with_cpu:
        sps, rounds, dt, npk = run_cpu(wl, cores, min_seconds=cpu_seconds, max_packets=40000)
        rec['cpu'] = {'value': sps, 'cores': cores, 'sample': f'{npk} packets x {rounds} passes in {dt:.1f} s'}
        rec['e2e_over_cpu'] = rec['e2e']['value'] / sps
    r.close()
    return rec


def library_record(pkg, torch, dev, rank, cores, steps, peak, dist, with_cpu):
    """The configs[4]-style library batch of this rank through the multi-track entry point (host buffers, pinned), and
    device-resident as one launch per bit depth."""
    import oracle_lib as ol
    tracks = build_library(rank, max(1, cores))
    lib = pkg.NewLibraryDecoder((dev,))
    pins, descs = [], []
    samples = comp = pcm_bytes = 0
    for t in tracks:
        fb = t['cfg'].frame_bytes()
        n = len(t['sizes'])
        pin_in = Pinned(pkg, len(t['packed']))
        pin_in.arr[:] = t['packed']
        pin_out = Pinned(pkg, n * fb)
        pins += [pin_in, pin_out]
        descs.append(pkg.Track(t['cookie'], pin_in.arr, t['offsets'], t['sizes']))
        t['out'] = pin_out.arr[:n * fb].reshape(n, fb)
        samples += t['frames'] * 2
        comp += int(t['sizes'].astype(np.int64).sum())
        pcm_bytes += t['frames'] * 2 * t['cfg'].bps()
    outs = [t['out'] for t in tracks]

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()

    res = lib.DecodeTracks(descs, out=outs)  # warm-up + gate: first and last track against the oracle, every status OK
    for t, r in zip(tracks, res):
        assert r.err is None and (r.status == 0).all()
    for t in (tracks[0], tracks[-1]):
        want, wnb, _ = ol.decode_batch(t['cfg'], t['packed'], t['offsets'][:32], t['sizes'][:32], nthreads=min(cores, 8))
        assert np.array_equal(t['out'][:32], want), 'library PCM differs from the oracle'
    lib.DecodeTracks(descs, out=outs)
    e2e_steps = max(2, min(steps, 4))
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        lib.DecodeTracks(descs, out=outs)
    e2e_s = time.perf_counter() - t0
    lib.close()
    # device-resident: the two depths as two stream-ordered launches
    groups = {}
    for t in tracks:
        groups.setdefault(t['bits'], []).append(t)
    runners = []
    for bits, ts in groups.items():
        packed = np.concatenate([t['packed'] for t in ts])
        base = np.cumsum([0] + [len(t['packed']) for t in ts])[:-1]
        offsets = np.concatenate([t['offsets'] + np.uint64(b) for t, b in zip(ts, base)])
        sizes = np.concatenate([t['sizes'] for t in ts])
        wl = dict(ts[0], packed=packed, offsets=offsets, sizes=sizes, frames=len(sizes) * 4096)
        r = Runner(pkg, torch, dev, wl)
        r.samples = sum(t['frames'] for t in ts) * 2
        r.gate(cores)
        runners.append(r)
    for r in runners:
        for _ in range(3):
            r.step_device()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0 = runners[0].stream
    for r in runners:
        r.stream = s0
    with torch.cuda.stream(s0):
        e0.record(s0)
        for _ in range(steps):
            for r in runners:
                r.step_device()
        e1.record(s0)
    barrier()
    ms_total = e0.elapsed_time(e1)
    for r in runners:
        r.close()
    rec = {'workload': LIB_DESC, 'tracks': len(tracks), 'packets': int(sum(len(t['sizes']) for t in tracks)), 'samples_per_step': samples,
           'ms_per_step': ms_total / steps, 'e2e_ms_per_step': e2e_s / e2e_steps * 1e3, 'compressed_bytes': comp, 'pcm_bytes': pcm_bytes,
           'gpu_launches_per_step': len(runners)}
    if with_cpu:
        t = tracks[1]
        sps, rounds, dt, npk = run_cpu(t, cores, min_seconds=2.0)
        t2 = tracks[0]
        sps2, rounds2, dt2, npk2 = run_cpu(t2, cores, min_seconds=2.0)
        rec['cpu'] = {'value': 2.0 / (1.0 / sps + 1.0 / sps2), 'cores': cores,
                      'sample': f'one 24-bit and one 16-bit track ({npk}+{npk2} packets) x {rounds}/{rounds2} passes, harmonic mean'}
    for p in pins:
        p.free()
    return rec


def api_legs(pkg, wl_c2, wl_c1, steps):
    """The drop-in API as a caller sees it, through the compiled C++ mirror (tools/api_bench.cpp)."""
    from m4a_writer import build_m4a
    exe = os.path.join(ROOT, 'tools', 'build', 'api_bench')  # built by build()
    src = os.path.join(ROOT, 'tools', 'api_bench.cpp')
    lib_dir = os.path.dirname(pkg.LIB_PATH)
    hdr = os.path.join(ROOT, 'saprobe-alac_b200', 'host', 'alac.hpp')
    out = {}
    with tempfile.TemporaryDirectory() as d:
        f = lambda n: os.path.join(d, n)
        if not os.path.exists(exe) or os.path.getmtime(exe) < max(os.path.getmtime(src), os.path.getmtime(hdr), os.path.getmtime(pkg.LIB_PATH)):
            exe = f('api_bench')  # missing or stale: compile a private copy, the tree may be read-only
            subprocess.run(['g++', '-std=c++17', '-O2', '-o', exe, src, '-L' + lib_dir, '-lalacb200', '-Wl,-rpath,' + lib_dir], check=True)
        open(f('cookie'), 'wb').write(wl_c2['cookie'])
        wl_c2['packed'].tofile(f('packed'))
        wl_c2['offsets'].astype(np.uint64).tofile(f('offs'))
        wl_c2['sizes'].astype(np.uint32).tofile(f('sizes'))
        r = subprocess.run([exe, 'packets', f('cookie'), f('packed'), f('offs'), f('sizes'), str(max(3, min(steps, 8)))], capture_output=True, text=True, timeout=600)
        if r.returncode == 0:
            dt, nbytes, _ = r.stdout.split()[:3]
            samples = wl_c2['frames'] * wl_c2['channels']
            assert int(nbytes) == samples * 3
            out['DecodePackets_c2'] = {'value': samples / float(dt), 'unit': 'samples/s', 'ms_per_call': float(dt) * 1e3,
                                       'how': 'alac::PacketDecoder::DecodePackets over all 14 063 packets ([]bytes in, fresh []bytes out), pageable caller '
                                              'memory, the decoder-owned pinned arena in between'}
        else:
            out['DecodePackets_c2'] = {'error': r.stderr[-300:]}
        packets = [bytes(wl_c1['packed'][int(o):int(o) + int(z)]) for o, z in zip(wl_c1['offsets'], wl_c1['sizes'])]
        data, _ = build_m4a(wl_c1['cookie'], packets, last_frames=wl_c1['frames'] % 4096)
        open(f('c1.m4a'), 'wb').write(data)
        r = subprocess.run([exe, 'read', f('c1.m4a'), str(max(5, min(steps, 20)))], capture_output=True, text=True, timeout=600)
        if r.returncode == 0:
            dt, nbytes, _, reuse = r.stdout.split()[:4]
            phases = [float(v) * 1e3 for v in r.stdout.split()[4:7]]
            samples = wl_c1['frames'] * wl_c1['channels']
            assert int(nbytes) == samples * 2
            out['NewDecoder_Read_c1'] = {'value': samples / float(dt), 'unit': 'samples/s', 'ms_per_file': float(dt) * 1e3,
                                         'x_realtime': wl_c1['seconds'] / float(dt), 'ms_per_file_decoder_kept_open': float(reuse) * 1e3,
                                         'ms_new_firstread_close': phases,
                                         'how': 'alac::Decoder::New + Read in 32 KiB pieces to EOF over the 60 s M4A (BASELINE configs[0]); the file '
                                                'image is pinned once and read in place, one GPU call per 2048-packet window'}
        else:
            out['NewDecoder_Read_c1'] = {'error': r.stderr[-300:]}
    return out


def main():
    # Libraries (NCCL's version banner, torchrun notices) may print to fd 1; the contract is one JSON line on stdout.
    # Everything else goes to stderr.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='c3', choices=sorted(WORKLOADS))
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--only-main', action='store_true', help='skip the sub-records (other configs, library batch, API legs)')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write what the timed path returned in its last step as DIR/*.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.warmup < 3 and args.impl == 'ours':
        args.warmup = 3

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    cores = host_cores()
    bits, ch, rate, seconds, desc = WORKLOADS[args.workload]
    config = {'workload': f'{args.workload}: {desc}', 'frame_length': 4096, 'encoder': 'test-side LPC encoder, orders 4-6',
              'signal': 'SURVEY 8d multi-sine + noise with silence / 2-LSB passages, seeded',
              'sharding': f'one batch cut into {world} contiguous packet ranges by shard_ranges (balanced by compressed bytes), one rank per GPU, no collective',
              'l2': 'inputs+outputs per step exceed the 126 MB L2 (no flush needed)'}

    # ------------------------------------------------------------------------------------------- reference arm
    if args.impl == 'reference':
        if rank != 0:
            return 0
        wl = build_workload(args.workload, seed=2, threads=cores)
        n = len(wl['sizes'])
        run_cpu(wl, cores, min_seconds=0.0, max_rounds=max(1, args.warmup))  # warm-up passes
        import oracle_lib as ol
        out = np.zeros((n, wl['cfg'].frame_bytes()), dtype=np.uint8)
        out[:] = 1
        t0 = time.perf_counter()
        for _ in range(args.steps):
            _, nb, st = ol.decode_batch(wl['cfg'], wl['packed'], wl['offsets'], wl['sizes'], nthreads=cores, out=out)
        dt = time.perf_counter() - t0
        if args.dump_outputs:
            idx = dump_index(n, wl)
            write_dump(args.dump_outputs, wl, idx, out[idx], nb, st)
        value = wl['frames'] * wl['channels'] * args.steps / dt
        line = {'impl': 'reference', 'metric': 'decoded PCM samples/s', 'value': value, 'unit': 'samples/s',
                'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': dt / args.steps * 1e3,
                'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'int32', 'data': 'synthetic',
                'config': config, 'x_realtime': value / ch / rate, 'frames_per_s': value / ch,
                'cpu_baseline': {'value': value, 'unit': 'samples/s', 'cores': cores, 'kind': 'port',
                                 'sample': f'whole workload ({n} packets) per step; C restatement of the Go reference '
                                           '(Go toolchain absent), thread per core over contiguous packet ranges'},
                'e2e': {'value': value, 'unit': 'samples/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
                'gpu_launches': 0}
        emit_line(line)
        return 0

    # ------------------------------------------------------------------------------------------------ our arm
    import torch
    from alac_b200_loader import load_package
    pkg = load_package()
    if not torch.cuda.is_available() or pkg.lib.alacb200_device_count() < 1:
        raise SystemExit('bench.py needs a CUDA device: the product path has no CPU fallback')
    dev = local_rank % torch.cuda.device_count()
    torch.cuda.set_device(dev)
    numa_node = bind_to_gpu_numa(dev) if world > 1 else None
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=torch.device('cuda', dev))

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # the ONE common batch: generated (or loaded from the cache) by rank 0 first, then read by the others
    if rank == 0:
        wl = build_workload(args.workload, seed=2, threads=cores)
    barrier()
    if rank != 0:
        wl = build_workload(args.workload, seed=2, threads=max(1, cores // world))
    lo, hi = pkg.shard_ranges(wl['sizes'], world)[rank]  # the product's partitioner
    run = Runner(pkg, torch, dev, wl, lo, hi)
    gate = run.gate(cores)

    sampler = ClockSampler(dev)
    sampler.start()
    ms_total, dec_ms, launches = run.time_device(args.steps, args.warmup, barrier)
    e2e_steps = max(3, min(args.steps, 10))
    e2e_s = run.time_host(e2e_steps, barrier)
    clocks = sampler.stop()
    barrier()
    if args.dump_outputs:  # the host leg writes its own buffers: the device buffers still hold the last timed step
        idx = dump_index(len(wl['sizes']), wl)
        parts = [run.device_results(idx[(idx >= lo) & (idx < hi)] - lo)]
        if dist is not None:
            mine, parts = parts[0], [None] * world
            dist.all_gather_object(parts, mine)  # contiguous shards in rank order: concatenation is batch order
        if rank == 0:
            write_dump(args.dump_outputs, wl, idx, *(np.concatenate([p[j] for p in parts]) for j in range(3)))
        barrier()

    # ---- max over ranks of the times, sums of the work -------------------------------------------------------------
    t = torch.tensor([ms_total, e2e_s * 1e3, dec_ms], dtype=torch.float64, device='cuda')
    h2d, d2h = run.bytes_per_step()
    w = torch.tensor([run.samples, run.comp_bytes, run.pcm_bytes, h2d, d2h, run.n], dtype=torch.float64, device='cuda')
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(w, op=dist.ReduceOp.SUM)
    ms_total, e2e_ms, dec_ms_max = (float(v) for v in t.cpu())
    samples, comp_bytes, pcm_bytes, h2d_all, d2h_all, n_all = (int(v) for v in w.cpu())
    value = samples * args.steps / (ms_total / 1e3)
    e2e_value = samples * e2e_steps / (e2e_ms / 1e3)
    peak, peak_src = measured_peak_gbs()
    traffic = None  # dram bytes of one launch from the committed ncu --set full capture of this workload
    try:
        with open(os.path.join(ROOT, 'profiles', 'latest_traffic.json')) as f:
            tj = json.load(f)
        if tj.get('workload') == args.workload and world == 1:
            traffic = tj['traffic_bytes_per_launch']
    except Exception:
        pass
    # roofline of the kernel as launched on THIS rank's shard (rank 0 reports its own launch)
    algo_bytes = run.comp_bytes + run.pcm_bytes
    achieved = algo_bytes / (dec_ms / 1e3) / 1e9

    line = {'metric': 'decoded PCM samples/s', 'value': value, 'unit': 'samples/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': ms_total / args.steps, 'higher_is_better': True, 'scaling': 'strong',
            'vs_baseline': None, 'dtype': 'int32', 'data': 'synthetic', 'config': config,
            'x_realtime': value / ch / rate, 'frames_per_s': value / ch,
            'e2e': {'value': e2e_value, 'unit': 'samples/s', 'h2d_bytes_per_step': h2d_all, 'd2h_bytes_per_step': d2h_all,
                    'ms_per_step': e2e_ms / e2e_steps, 'steps': e2e_steps, 'x_realtime': e2e_value / ch / rate,
                    'how': 'alacb200_decode_packets on pinned host buffers, host clock around the blocking call, max over ranks'},
            'gpu_launches': launches,
            'kernels_ms_per_step': {'alac_decode_kernel': dec_ms},
            'roofline': {'bound': 'hbm', 'kernel': 'alac_decode_kernel', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s',
                         'frac': achieved / peak, 'traffic': traffic, 'peak_source': peak_src,
                         'algorithmic_bytes_per_launch': algo_bytes,
                         'note': 'compressed bytes read once + PCM bytes written once per packet (SURVEY 8d) over the one '
                                 'kernel of the path (entropy + predictor + emit), one launch per step; ALU-pipe / latency-bound, see profiles/'},
            'clocks': clocks, 'packets': n_all, 'packets_this_rank': run.n, 'compressed_bytes': comp_bytes, 'pcm_bytes': pcm_bytes,
            'host_cores': cores, 'numa_node': numa_node,
            'gate': f'{gate} packets per workload checked against the oracle before timing; the full-size bit-exact checks are tests/test_gpu_parity.py '
                    'and tests/test_gpu_library.py'}

    with_cpu = rank == 0 and not args.no_cpu_baseline and world == 1
    if with_cpu:
        sps, rounds, dt, npk = run_cpu(wl, cores, min_seconds=8.0)
        line['cpu_baseline'] = {'value': sps, 'unit': 'samples/s', 'cores': cores, 'kind': 'port',
                                'sample': f'whole workload ({npk} packets) x {rounds} passes in {dt:.1f} s; C restatement of the '
                                          'Go reference (no Go toolchain in the image), one thread per core'}
    run.close()

    if not args.only_main:
        sub_steps = max(3, min(args.steps, 10))
        # ---- the library batch, one track list per rank (weak scaling of the multi-track path) ----------------------
        lw = library_record(pkg, torch, dev, rank, cores, sub_steps, peak, dist, with_cpu)
        tt = torch.tensor([lw['ms_per_step'], lw['e2e_ms_per_step']], dtype=torch.float64, device='cuda')
        ww = torch.tensor([lw['samples_per_step'], lw['tracks'], lw['packets'], lw['compressed_bytes'] + lw['pcm_bytes']], dtype=torch.float64, device='cuda')
        if dist is not None:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dist.all_reduce(ww, op=dist.ReduceOp.SUM)
        lms, lems = (float(v) for v in tt.cpu())
        lsamples, ltracks, lpackets, lbytes = (int(v) for v in ww.cpu())
        lib_rec = {'workload': LIB_DESC, 'scaling': 'weak', 'tracks': ltracks, 'packets': lpackets,
                   'value': lsamples / (lms / 1e3), 'unit': 'samples/s', 'ms_per_step': lms,
                   'e2e': {'value': lsamples / (lems / 1e3), 'ms_per_step': lems,
                           'how': 'alacb200_library_decode_tracks, pinned track buffers read in place, max over ranks'},
                   'roofline_frac': lbytes / world / (lms / 1e3) / 1e9 / peak, 'gpu_launches_per_step': lw['gpu_launches_per_step']}
        if 'cpu' in lw:
            lib_rec['cpu'] = lw['cpu']
            lib_rec['e2e_over_cpu'] = lib_rec['e2e']['value'] / lw['cpu']['value']
        line['lib_weak'] = lib_rec
        if world == 1 and rank == 0:
            subs = {}
            wls = {}
            for name, seed in (('c1', 1), ('c2', 2), ('c4', 4)):
                if name == args.workload:
                    continue
                wls[name] = build_workload(name, seed=seed, threads=cores)
                subs[name] = sub_record(pkg, torch, dev, wls[name], cores, sub_steps, peak, with_cpu=with_cpu)
            ffw = build_ffmpeg_workload()
            if ffw is not None:
                subs['c2_ffmpeg'] = sub_record(pkg, torch, dev, ffw, cores, sub_steps, peak, with_cpu=False)
                subs['c2_ffmpeg']['encoder'] = "FFmpeg 8 libavcodec 'alac' encoder (defaults) on the same signal as c2"
            subs['lib'] = lib_rec
            line['workloads'] = subs
            if 'c2' in wls and 'c1' in wls:
                try:
                    line['e2e_api'] = api_legs(pkg, wls['c2'], wls['c1'], sub_steps)
                except Exception as e:  # a missing compiler must not lose the line
                    line['e2e_api'] = {'error': str(e)[:200]}
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        emit_line(line)
    return 0


if __name__ == '__main__':
    sys.exit(main())
