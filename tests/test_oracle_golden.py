"""The CPU oracle against the committed golden vectors (SURVEY.md section 8c).

Every fixture was produced by FFmpeg's independent ALAC encoder and verified at generation time to
decode to the source PCM with FFmpeg's decoder; here the oracle must reproduce the recorded sha256
of that source PCM -- the same bit-for-bit check as tests/conformance_test.go:282-292.
"""
import hashlib

import numpy as np
import pytest

import oracle_lib as ol
from golden_io import load_fixtures
from signals import make_signal

FIX = load_fixtures()


@pytest.mark.parametrize('name', sorted(FIX))
def test_oracle_matches_ffmpeg_golden(name):
    fx = FIX[name]
    m = fx['meta']
    st, cfg = ol.parse_cookie(fx['cookie'])
    assert st == ol.OK
    assert (cfg.bit_depth, cfg.num_channels, cfg.sample_rate) == (m['bits'], m['channels'], m['sample_rate'])
    pcm = b''
    for p in fx['packets']:
        st, out = ol.decode_packet(cfg, p)
        assert st == ol.OK
        pcm += out
    assert len(pcm) == m['frames'] * m['channels'] * cfg.bps()
    assert hashlib.sha256(pcm).hexdigest() == m['pcm_sha256']


@pytest.mark.parametrize('name', ['s16_stereo_44k', 's24_71_48k', 's16_stereo_silence_lsb'])
def test_golden_source_is_reproducible(name):
    """The recorded hash really is the seeded source signal (format-metadata check, conformance_test.go:267-279)."""
    m = FIX[name]['meta']
    x = make_signal(m['kind'], m['channels'], m['frames'], m['bits'], m['sample_rate'], seed=m['seed'])
    assert hashlib.sha256(ol.int_to_pcm_bytes(x, m['bits'])).hexdigest() == m['pcm_sha256']


def test_batch_driver_equals_single(fixtures=None):
    fx = FIX['s24_stereo_96k']
    st, cfg = ol.parse_cookie(fx['cookie'])
    packed, offs, sizes = ol.pack(fx['packets'])
    out, nb, status = ol.decode_batch(cfg, packed, offs, sizes, nthreads=3)
    assert (status == 0).all()
    for i, p in enumerate(fx['packets']):
        st, pcm = ol.decode_packet(cfg, p)
        assert bytes(out[i, :nb[i]]) == pcm


def test_encoder_roundtrip_all_depths():
    """test-side encoder -> oracle == source for the depths FFmpeg cannot make (restatement only)."""
    for bits, shift in ((20, 0), (32, 2), (24, 0), (24, 2), (16, 0)):
        for ch in (1, 2, 6):
            cfg = ol.Config.make(bit_depth=bits, num_channels=ch, sample_rate=48000)
            x = make_signal('silence_lsb', ch, 5000, bits, 48000, seed=bits + ch)
            pk = ol.encode_stream(cfg, x, ol.PacketOpts.make(bytes_shifted=shift))
            got = []
            for p in pk:
                st, pcm = ol.decode_packet(cfg, p)
                assert st == ol.OK
                got.append(ol.pcm_bytes_to_int(pcm, bits, ch))
            y = np.concatenate(got)
            if bits == 20:
                y = y >> 4
            assert np.array_equal(y, x), (bits, shift, ch)


def test_synthetic_cases_are_well_formed_for_the_oracle():
    """The synthetic suites the GPU parity tests use: exotic cases decode (or hit a reference panic), hostile packets end in one of the
    reference's sentinels (or where it would panic), and the threaded batch driver equals packet-by-packet decoding."""
    import synth_cases
    n_exotic = n_hostile = 0
    for name, cfg, packets in synth_cases.exotic_cases() + synth_cases.frame_length_cases() + synth_cases.entropy_edge_cases():
        for p in packets:
            st, pcm = ol.decode_packet(cfg, p)
            assert (pcm is None) == (st != ol.OK), name
            # the only exotic shapes that do not decode are the ones on which the reference panics (appendix B7)
            assert st == ol.OK or ol.code(st) == 9, (name, st)
            n_exotic += st == ol.OK
    seen = set()
    for name, cfg, packets in synth_cases.hostile_cases(max_per_seed=12):
        packed, offs, sizes = ol.pack(packets)
        out, nb, status = ol.decode_batch(cfg, packed, offs, sizes, nthreads=3)
        for i, p in enumerate(packets):
            n_hostile += 1
            st, pcm = ol.decode_packet(cfg, p)
            assert st == status[i], name
            assert (pcm is None) == (st != ol.OK), name
            if pcm is not None:
                assert bytes(out[i, :nb[i]]) == pcm, name
            seen.add(ol.code(st))
    assert n_exotic > 200 and n_hostile > 300
    assert seen <= {0, 3, 4, 5, 6, 7, 9}, seen


def test_wide_ffmpeg_matrix_oracle():
    """The reference's own conformance matrix (conformance_test.go:573-628: {16, 24} x 11 rates x 1-8 channels; here 64
    packets + a partial one at three of the rates, 3 packets at the others), FFmpeg-encoded on the spot:
    oracle == FFmpeg-decode == source, bit for bit, and the format metadata of the cookie (conformance_test.go:267-279)."""
    import os, sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden'))
    import wide_matrix
    if not wide_matrix.ffmpeg_available():
        pytest.skip('FFmpeg libraries (opencv_python_headless.libs) not importable here; ffmpeg_fixtures.npz remains the pin')
    npk = 0
    for case in wide_matrix.wide_cases():
        cookie, packets, x = wide_matrix.build(case)
        st, cfg = ol.parse_cookie(cookie)
        assert st == ol.OK and (cfg.bit_depth, cfg.num_channels, cfg.sample_rate) == (case['bits'], case['channels'], case['rate'])
        packed, offs, sizes = ol.pack(packets)
        out, nb, status = ol.decode_batch(cfg, packed, offs, sizes, nthreads=4)
        assert (status == 0).all(), case['name']
        got = b''.join(bytes(out[i, :nb[i]]) for i in range(len(packets)))
        assert got == ol.int_to_pcm_bytes(x, case['bits']), case['name']
        npk += len(packets)
    assert npk > 3000


def test_exotic_ffmpeg_matrix_oracle():
    """What FFmpeg's encoder never emits but its decoder reads (tests/golden/exotic_matrix.py: 20- and 32-bit, 0 / 1 / 2
    shifted bytes, the order-31 pre-pass, orders 0-31; streams from the test-side encoder): FFmpeg-decode == source is
    asserted in build() (or was, for the committed list of confirmed cases), here oracle == source. An independent pin for
    shapes that were restatement-only."""
    import os, sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden'))
    import exotic_matrix
    confirmed, depths = 0, set()
    for case, cfg, packets, x in exotic_matrix.checked_cases():
        packed, offs, sizes = ol.pack(packets)
        out, nb, status = ol.decode_batch(cfg, packed, offs, sizes, nthreads=4)
        assert (status == 0).all(), case['name']
        got = b''.join(bytes(out[i, :nb[i]]) for i in range(len(packets)))
        assert got == ol.int_to_pcm_bytes(x, case['bits']), case['name']
        confirmed += 1
        depths.add((case['bits'], case['shift'], case['mode']))
    assert confirmed >= 300 and {(20, 0, 0), (20, 0, 15), (24, 0, 0), (24, 1, 15), (32, 1, 0), (32, 2, 0), (32, 2, 15), (16, 0, 15)} <= depths


def test_synth_hashes_pin_the_oracle():
    """Drift pin for the restatement-only cases (20/32-bit, mode != 0, odd orders, DSE/FIL, hostile statuses ...): the
    oracle's status word, byte count and PCM of every synthetic case must equal tests/golden/synth_hashes.json, recorded
    when the oracle was cross-checked (gen_synth_hashes.py). The GPU suite asserts the same table, so kernel and oracle
    cannot drift together. A case whose generated INPUT differs from the recorded one (the seeded signals go through
    libm; another CPU may round one sample differently) is not judged; there must be next to none of them."""
    import synth_pin
    pin = synth_pin.load_pin()['cases']
    cases = synth_pin.all_cases()
    assert {n for n, _, _ in cases} == set(pin), 'case list changed: regenerate tests/golden/synth_hashes.json and say why'
    other_input, bad = [], []
    for name, cfg, packets in cases:
        if synth_pin.packets_digest(cfg, packets) != pin[name]['packets_sha256']:
            other_input.append(name)
            continue
        st, nb, out = synth_pin.oracle_result(cfg, packets)
        if synth_pin.result_digest(st, nb, out) != pin[name]['result_sha256']:
            bad.append(name)
    assert not bad, f'oracle output drifted on {len(bad)} cases: {bad[:5]}'
    assert len(other_input) <= len(cases) // 20, f'{len(other_input)} cases generate other inputs here: {other_input[:5]}'


def test_oracle_under_address_sanitizer(tmp_path):
    """The oracle compiled with AddressSanitizer + UBSan over the exotic and hostile suites (every packet and every output
    buffer in an exact-size heap block): no access outside either, and the same status / byte count / PCM hash as the
    regular build. The places where the Go reference would panic must come back as status 9, not as memory errors."""
    import os, subprocess, synth_cases
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    probe = tmp_path / 'probe.c'
    probe.write_text('int main(void){return 0;}')
    if subprocess.run(['gcc', '-fsanitize=address,undefined', '-o', str(tmp_path / 'probe'), str(probe)], capture_output=True).returncode != 0:
        pytest.skip('no sanitizer runtime in this image')
    exe = str(tmp_path / 'oracle_asan')
    # signed overflow is defined here (-fwrapv, as in oracle/Makefile); the shift checks stay on: Go's shift semantics are explicit in the source
    subprocess.run(['gcc', '-O1', '-g', '-fwrapv', '-fsanitize=address,undefined', '-fno-sanitize=signed-integer-overflow',
                    '-fno-sanitize-recover=undefined', '-o', exe, os.path.join(root, 'tests', 'cpp', 'oracle_asan_driver.c'),
                    os.path.join(root, 'oracle', 'alac_oracle.c'), '-lpthread'], check=True)
    blob = tmp_path / 'cases.bin'
    want = []
    with open(blob, 'wb') as f:
        def put(cfg, packets):
            cookie = ol.make_cookie(cfg)
            f.write(len(cookie).to_bytes(4, 'little') + cookie + len(packets).to_bytes(4, 'little'))
            for p in packets:
                f.write(len(p).to_bytes(4, 'little') + bytes(p))
                st, pcm = ol.decode_packet(cfg, p)
                h = 2166136261
                for b in (pcm or b''):
                    h = ((h ^ b) * 16777619) & 0xffffffff
                want.append(f'{st} {len(pcm or b"")} {h}')
        for name, cfg, packets in synth_cases.exotic_cases():
            put(cfg, packets[:2])
        for name, cfg, packets in synth_cases.frame_length_cases() + synth_cases.entropy_edge_cases():
            if cfg.frame_length <= 4097:
                put(cfg, packets)
        for name, cfg, packets in synth_cases.hostile_cases(max_per_seed=10):
            put(cfg, packets)
    r = subprocess.run([exe, str(blob)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    got = r.stdout.split('\n')[:-1]
    assert len(got) == len(want) and len(want) > 500
    bad = [i for i, (a, b) in enumerate(zip(got, want)) if a != b]
    assert not bad, (bad[:5], [got[i] for i in bad[:3]], [want[i] for i in bad[:3]])
