"""Shapes FFmpeg's ALAC ENCODER never emits but its DECODER reads: a second, independent pin for them.

The test-side encoder (oracle/alac_encoder.c) produces 20- and 32-bit streams, every `bytesShifted` a depth allows, the
order-31 pre-pass (`mode` 15 -- the one non-zero mode FFmpeg implements; the Go reference runs the pre-pass for ANY
non-zero mode, decoder.go:306-308), predictor orders 0-31, parameter sweeps, other frame lengths, escape elements, the LFE
tag and partial-frame headers. build(case) asserts that FFmpeg's decoder returns the
source PCM for the packets; the tests then require the same of the oracle (tests/test_oracle_golden.py, CPU) and of the
CUDA path (tests/test_gpu_parity.py). Before this matrix those shapes were compared with the restatement only.

Left out because FFmpeg and the Go reference legitimately differ, or FFmpeg refuses: negative mixRes (FFmpeg reads it
unsigned, decoder.go:422 sign-extends), denShift 14-15 / coefficients at the int16 limit (FFmpeg wraps coefficients at
16 bits for every order, predictor.go:107-110 keeps int32 for orders 4/5/6/8: a denShift-14 stream of this generator
decodes differently there), modes other than 0 and 15, mixing weights above 1 (mixRes >= 1 << mixBits), which push U past its channel width on loud material: the values
wrap at chanBits and the FIR sum can leave int32, where FFmpeg's arithmetic and the reference's differ, and elements
whose sample width exceeds 32 bits (32-bit pairs without shifted bytes, 32-bit escape pairs: "bps 33 is not
implemented"), DSE / FIL elements and packets without an END tag (FFmpeg refuses them): build() returns None for a case
FFmpeg rejects.

The names of the cases FFmpeg confirmed are committed (exotic_confirmed.json, `python tests/golden/exotic_matrix.py`
rewrites it), so that checked_cases() still yields those streams -- all of them from the test-side encoder and seeds --
where the FFmpeg libraries are not installed.
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
CONFIRMED_PATH = os.path.join(HERE, 'exotic_confirmed.json')
sys.path.insert(0, os.path.dirname(HERE))
import oracle_lib as ol  # noqa: E402
from signals import make_signal  # noqa: E402

KINDS = ('music', 'silence_lsb', 'loud')
ORDERS = ((4, 6), (8, 8), (1, 30), (0, 0), (31, 31))


def exotic_cases():
    """-> list of dict(name, bits, channels, shift, mode, orders, kind, frames, seed)"""
    out, seed = [], 7000
    for bits, shifts in ((20, (0,)), (32, (1, 2)), (24, (0, 1)), (16, (0,))):
        for ch in (1, 2, 3, 6, 8):
            for shift in shifts:
                for mode in (0, 15):
                    if bits in (16, 24) and mode == 0 and shift == (1 if bits == 24 else 0):
                        continue  # what FFmpeg's encoder emits itself: wide_matrix.py
                    for oi, orders in enumerate(ORDERS):
                        seed += 1
                        out.append(dict(name=f'x{bits}_c{ch}_s{shift}_m{mode}_o{orders[0]}-{orders[1]}', bits=bits, channels=ch, shift=shift,
                                        mode=mode, orders=orders, kind=KINDS[(oi + ch + shift + mode) % 3], frames=2 * 4096 + 777 + ch, seed=seed))
    # pbFactor / denShift / mixBits / non-negative mixRes sweeps on pairs at every depth (FFmpeg reads mixRes unsigned)
    for bits, shift in ((16, 0), (20, 0), (24, 1), (24, 0), (32, 2)):
        for (pbf, den, mb_, mr) in ((4, 9, 0, 0), (2, 7, 2, 1), (7, 12, 2, 3), (1, 4, 5, 3), (4, 9, 31, 1), (3, 11, 8, 100), (5, 10, 7, 127)):
            seed += 1
            out.append(dict(name=f'x{bits}_s{shift}_pb{pbf}_den{den}_mix{mb_}-{mr}', bits=bits, channels=2, shift=shift, mode=0, orders=(4, 8),
                            kind=KINDS[seed % 3], frames=4096 + 555, seed=seed, pb_factor=pbf, den_shift=den, mix_bits=mb_, mix_res=mr))
    # frame lengths other than 4096 (the cookie's frameLength, config.go:27-38)
    for fl in (256, 1024, 8192):
        for bits, shift in ((16, 0), (20, 0), (24, 1), (32, 2)):
            for ch in (1, 2, 6):
                seed += 1
                out.append(dict(name=f'x{bits}_c{ch}_fl{fl}', bits=bits, channels=ch, shift=shift, mode=0, orders=(4, 6), kind=KINDS[seed % 3],
                                frames=3 * fl + fl // 3 + ch, seed=seed, frame_length=fl))
    # escape (uncompressed) elements, the LFE tag, the partial-frame header on every packet
    for opt in ('force_escape', 'lfe_tag3', 'always_partial'):
        for bits, shift in ((16, 0), (20, 0), (24, 1), (32, 2)):
            for ch in (1, 2, 6):
                seed += 1
                out.append(dict(name=f'x{bits}_c{ch}_{opt}', bits=bits, channels=ch, shift=shift, mode=0, orders=(4, 6), kind=KINDS[seed % 3],
                                frames=2 * 4096 + 300 + ch, seed=seed, **{opt: 1}))
    return out


def ffmpeg_available():
    try:
        sys.path.insert(0, HERE)
        import ffmpeg_alac  # noqa: F401
        return True
    except Exception:
        return False


def encode(case):
    """-> (oracle config, [packets], source int64 [frames, ch]) from the test-side encoder, or None when it has no
    representation for a frame (a 32-bit pair that needs an escape element)."""
    rate = 48000
    x = make_signal(case['kind'], case['channels'], case['frames'], case['bits'], rate, seed=case['seed'])
    cfg = ol.Config.make(bit_depth=case['bits'], num_channels=case['channels'], sample_rate=rate, frame_length=case.get('frame_length', 4096))
    extra = {k: case[k] for k in ('pb_factor', 'den_shift', 'mix_bits', 'mix_res', 'force_escape', 'lfe_tag3', 'always_partial') if k in case}
    opts = ol.PacketOpts.make(min_order=case['orders'][0], max_order=case['orders'][1], bytes_shifted=case['shift'], mode=case['mode'], **extra)
    try:
        return cfg, ol.encode_stream(cfg, x, opts), x
    except ValueError:
        return None


def build(case):
    """-> (oracle config, [packets], source int64 [frames, ch]) after FFmpeg's decoder has returned the source for these
    packets, or None when FFmpeg rejects the stream (sample width above 32 bits)."""
    sys.path.insert(0, HERE)
    import ffmpeg_alac as ff
    built = encode(case)
    if built is None:
        return None
    cfg, packets, x = built
    rate = cfg.sample_rate
    try:
        y = ff.alac_decode(ol.make_cookie(cfg, wrappers=1), packets, case['bits'], case['channels'], rate).T
    except (RuntimeError, ValueError):  # send_packet refused, or no frame came out
        return None
    if y.shape != x.shape:
        return None
    assert np.array_equal(y, x), f"FFmpeg's decoder does not return the source for {case['name']}"
    return cfg, packets, x


def checked_cases():
    """-> [(case, cfg, packets, source)] of the streams FFmpeg's decoder returns the source for: confirmed now when the
    FFmpeg libraries are present, else the committed list of confirmed cases."""
    if ffmpeg_available():
        built = ((case, build(case)) for case in exotic_cases())
    else:
        with open(CONFIRMED_PATH) as f:
            names = set(json.load(f)['cases'])
        built = ((case, encode(case)) for case in exotic_cases() if case['name'] in names)
    return [(case, *b) for case, b in built if b is not None]


if __name__ == '__main__':
    assert ffmpeg_available(), 'confirming the cases needs the FFmpeg libraries'
    names = [case['name'] for case, _, _, _ in checked_cases()]
    with open(CONFIRMED_PATH, 'w') as f:
        json.dump(dict(what="exotic_matrix cases whose packets FFmpeg's ALAC decoder (libavcodec 62.11.100) decodes to the source",
                       cases=names), f, indent=0)
    print(len(names), 'cases confirmed')
