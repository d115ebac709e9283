"""CPU: which VBZ zstd frames the host hands to the device decoder (fast5.zstd_frame_size), the stored form of a
read (fast5.stored_chunks) and the header-level inspector the device tests measure their coverage with."""
import numpy as np
import pytest

import _h5write as hw
import _zstd as Z
from oracle import zstd_inspect
from warpstr_b200 import fast5

DATA = b''.join(bytes([i % 7, i % 13]) for i in range(30000))


@pytest.mark.parametrize('level', Z.LEVELS)
def test_plain_frames_go_to_the_device(level):
    f = Z.compress(DATA, level)
    assert fast5.zstd_frame_size(f, len(DATA)) == len(DATA) == Z.content_size(f)
    assert fast5.zstd_frame_size(f, len(DATA) - 1) == -1                      # above the host decoder's bound


@pytest.mark.parametrize('n', [1, 255, 256, 65791, 65792, 300000])
def test_every_content_size_field(n):
    data = bytes(range(256)) * (n // 256 + 1)
    f = Z.compress(data[:n], 3)
    assert fast5.zstd_frame_size(f, n) == n
    assert zstd_inspect.inspect(f)['fcs_bytes'] == (1 if n < 256 else 2 if n < 65792 else 4)


def test_frames_the_device_does_not_take():
    ok = Z.compress(DATA, 1)
    checksummed = Z.compress(DATA, 1, checksum=True)
    no_size = Z.compress(DATA, 1, content_size=False)
    assert zstd_inspect.inspect(checksummed)['checksum'] and Z.content_size(no_size) == -1
    skippable = (0x184D2A50).to_bytes(4, 'little') + (3).to_bytes(4, 'little') + b'abc'
    for f in (checksummed, no_size, ok + ok, ok + skippable, skippable + ok, ok[:-1], ok + b'\0', b'', ok[:8]):
        assert fast5.zstd_frame_size(f, 10 ** 7) == -1
    with_dict = bytearray(ok)
    with_dict[4] |= 1                                        # a dictionary ID field
    assert fast5.zstd_frame_size(bytes(with_dict), 10 ** 7) == -1


def test_classifier_agrees_with_the_headers():
    for name, f, content in Z.corpus() + Z.hand_frames():
        info = zstd_inspect.inspect(f)
        assert info['end'] == len(f) and not info['checksum'], name
        assert fast5.zstd_frame_size(f, len(content)) == len(content) == Z.content_size(f), name


def _reads(seed=0):
    rng = np.random.default_rng(seed)
    return {f'{i:02d}-r': (450 + np.cumsum(rng.integers(-50, 51, size=n))).astype(np.int16)
            for i, n in enumerate([1, 999, 4097, 10001])}


@pytest.mark.parametrize('filt', ['vbz0', 'vbz1', 'vbz0-raw', 'vbz1-raw', 'vbz0-nozz', 'deflate', 'none',
                                  'contiguous'])
def test_stored_chunks_decode_to_the_signal(tmp_path, filt):
    reads = _reads()
    p = str(tmp_path / 'm.fast5')
    hw.write_multi(p, reads, filt, chunk=1000)
    for rid, x in reads.items():
        sc = fast5.stored_chunks(p, rid)
        rc = fast5.raw_chunks(p, rid)
        assert np.array_equal(sc.decode(), fast5.raw_signal(p, rid)) and np.array_equal(sc.decode(), x)
        assert [c.start for c in sc.chunks] == [c.start for c in rc.chunks]
        zstd = filt in ('vbz0', 'vbz1', 'vbz0-nozz')
        for s, r in zip(sc.chunks, rc.chunks):
            if zstd:
                assert s.kind == r.kind + fast5.KIND_VBZ0_ZSTD and s.body_size == len(r.payload)
                assert Z.reference(s.payload, s.body_size) == r.payload
            else:
                assert s == r
            assert s.unzstd() == r


def test_stored_chunks_keep_checksummed_frames_on_the_host(tmp_path, monkeypatch):
    reads = _reads(1)
    p = str(tmp_path / 'c.fast5')
    monkeypatch.setattr(hw, 'zstd_compress', lambda body, level=1: Z.compress(body, level, checksum=True))
    hw.write_multi(p, reads, 'vbz1', chunk=1000)
    for rid, x in reads.items():
        sc = fast5.stored_chunks(p, rid)
        assert {c.kind for c in sc.chunks} == {fast5.KIND_VBZ1}
        assert np.array_equal(sc.decode(), x)


def test_inspector_reports_block_and_section_kinds():
    seen = set()
    for _, f, _ in Z.corpus() + Z.hand_frames():
        for b in zstd_inspect.inspect(f)['blocks']:
            seen.add(b['type'])
            if b['type'] == 'compressed':
                seen.add((b['literals'], b['streams']))
    assert {'raw', 'rle', 'compressed', ('raw', 1), ('rle', 1), ('huffman', 1), ('huffman', 4)} <= seen
