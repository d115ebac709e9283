"""GPU: zstd frames decoded on the device (wstr_zstd_decode_batch) against libzstd, byte for byte, and the fast5
route that sends VBZ chunks as their files store them (fast5.stored_chunks -> pack_vbz -> call_arrays_vbz /
locate_arrays_vbz / main_wrapper) against the route that undoes zstd on the host."""
import os
import struct

import numpy as np
import pytest

import _h5write as hw
import _zstd as Z
from oracle import zstd_inspect
from warpstr_b200 import fast5, synth

pytestmark = pytest.mark.gpu
GUARD = 0xA5
CORRUPT = 5          # WSTR_ZSTD_CORRUPT


def _decode(frames, sizes):
    """Every frame in one call: frames at 16-byte aligned offsets, the last one with only its padding behind it
    in the input buffer; outputs apart by 7 guard bytes, which must come back untouched.  -> (outputs, status)"""
    import torch
    from warpstr_b200 import _lib
    m = len(frames)
    in_bytes = np.array([len(f) for f in frames], dtype=np.int64)
    in_off = np.zeros(m, dtype=np.int64)
    in_off[1:] = np.cumsum((in_bytes[:-1] + 15) & ~15)
    pay = np.zeros(int(in_off[-1] + ((in_bytes[-1] + 15) & ~15)), dtype=np.uint8)
    for f, o in zip(frames, in_off):
        pay[o:o + len(f)] = np.frombuffer(f, dtype=np.uint8)
    out_bytes = np.array(sizes, dtype=np.int64)
    out_off = np.zeros(m, dtype=np.int64)
    out_off[1:] = np.cumsum(out_bytes[:-1] + 7)
    total = int(out_off[-1] + out_bytes[-1]) + 7
    d_out = torch.full((total,), GUARD, dtype=torch.uint8, device='cuda')
    d_status = torch.full((m,), -7, dtype=torch.int32, device='cuda')
    ws = torch.empty(_lib.zstd_workspace_bytes(m), dtype=torch.uint8, device='cuda')
    _lib.zstd_decode_batch(torch.from_numpy(pay).cuda(), in_off, in_bytes, out_off, out_bytes, d_out, d_status, ws)
    out = d_out.cpu().numpy()
    inside = np.zeros(total, dtype=bool)
    for o, n in zip(out_off, out_bytes):
        inside[o:o + n] = True
    assert (out[~inside] == GUARD).all(), 'a frame wrote outside its output range'
    return [out[o:o + n].tobytes() for o, n in zip(out_off, out_bytes)], d_status.cpu().numpy()


@pytest.fixture(scope='module')
def corpus():
    frames = Z.corpus() + Z.hand_frames()
    for name, f, content in frames:
        assert Z.reference(f, len(content)) == content, name        # hand-built frames included
    return frames


def test_corpus_matches_libzstd(built_lib, corpus):
    outs, st = _decode([f for _, f, _ in corpus], [len(c) for _, _, c in corpus])
    for (name, _, content), got, s in zip(corpus, outs, st):
        assert s == 0, (name, s)
        assert got == content, name


def test_corpus_covers_every_section_kind(corpus):
    seen = set()
    for _, f, _ in corpus:
        info = zstd_inspect.inspect(f)
        seen.add(('fcs', info['fcs_bytes']))
        for b in info['blocks']:
            seen.add(('block', b['type']))
            if b['type'] == 'compressed':
                seen.add(('literals', b['literals'], b['streams']))
                for k, v in (b['modes'] or {}).items():
                    seen.add((k, v))
    want = {('fcs', 1), ('fcs', 2), ('fcs', 4), ('block', 'raw'), ('block', 'rle'), ('block', 'compressed')}
    want |= {('literals', t, s) for t in ('huffman', 'treeless') for s in (1, 4)}
    want |= {('literals', 'raw', 1), ('literals', 'rle', 1)}
    want |= {(k, v) for k in ('LL', 'OF', 'ML') for v in zstd_inspect.MODES}
    assert want <= seen, sorted(want - seen)


def _in_four_stream_literals(frame, byte):
    return any(b.get('streams') == 4 and b['huf_streams'][0] <= byte < b['huf_streams'][1]
               for b in zstd_inspect.inspect(frame)['blocks'])


def _sets_reserved_mode_bits(frame, damaged, byte):
    """The flip set a reserved bit of a sequences modes byte, which libzstd checks only from 1.5.6 on."""
    return any(b.get('modes_at') == byte for b in zstd_inspect.inspect(frame)['blocks']) and damaged[byte] & 3


def test_corruption_statuses_match_libzstd(built_lib, corpus):
    """Truncations and single-bit flips spread over every corpus frame.  The device refuses a frame exactly
    where libzstd does, and agrees byte for byte where both decode it.  Two documented differences, where the
    device follows RFC 8878 and libzstd accepts (WSTR_ZSTD_CORRUPT): libzstd's fast four-stream Huffman loops
    (x86-64 with BMI2) skip the check that each stream is consumed exactly, and libzstd before 1.5.6 ignores
    the reserved bits of the sequences modes byte."""
    rng = np.random.default_rng(7)
    frames, sizes, cases = [], [], []
    for k in range(2400):
        name, f, content = corpus[k % len(corpus)]
        b = bytearray(f)
        if k % 8 == 0:
            cut = int(rng.integers(1, len(b)))
            b, byte = b[:cut], -1
        else:
            pos = int(rng.integers(len(b) * 8))
            b[pos // 8] ^= 1 << (pos % 8)
            byte = pos // 8
        frames.append(bytes(b))
        sizes.append(len(content))
        cases.append((name, f, byte))
    outs, st = _decode(frames, sizes)
    refused = lax = 0
    for (name, f, byte), fr, size, got, s in zip(cases, frames, sizes, outs, st):
        want = Z.reference(fr, size)
        if want is None:
            assert s != 0, (name, byte)
            refused += 1
        elif s != 0:
            assert s == CORRUPT and byte >= 0, (name, byte, s)
            assert _in_four_stream_literals(f, byte) or (Z.version() < 10506 and
                                                         _sets_reserved_mode_bits(f, fr, byte)), (name, byte)
            lax += 1
        else:
            assert got == want, (name, byte)
    assert refused > 500 and lax < 0.1 * len(cases)


def test_calls_without_frames_and_bad_arguments(built_lib):
    import torch
    from warpstr_b200 import _lib
    ws = torch.empty(_lib.zstd_workspace_bytes(1), dtype=torch.uint8, device='cuda')
    d = torch.zeros(64, dtype=torch.uint8, device='cuda')
    st = torch.zeros(1, dtype=torch.int32, device='cuda')
    _lib.zstd_decode_batch(d, [], [], [], [], d, st, ws)
    with pytest.raises(_lib.WarpstrError):                  # misaligned frame
        _lib.zstd_decode_batch(d, [8], [9], [0], [1], d, st, ws)
    with pytest.raises(_lib.WarpstrError):
        _lib.zstd_decode_batch(d, [0], [9], [0], [1], d, st, ws[:8])


# -- the fast5 route ----------------------------------------------------------------------------------------
def _mixed_reads(n_reads, seed):
    """Synthetic HD reads whose chunks are zstd frames, StreamVByte bodies or raw int16, mixed in every read;
    -> (reads with frames, the same reads with every frame undone on the host, windows, strands)."""
    locus = synth.make_locus('HD', seed=seed)
    reads = synth.make_reads(locus, n_reads, seed=seed + 1, noise=0.2)
    rng = np.random.default_rng(seed + 2)
    stored, hosted, wins = [], [], []
    for i, r in enumerate(reads):
        x, lo, hi = synth.to_raw_int16(rng, r.signal, pad=int(rng.integers(100, 3000)), spike_rate=5e-4)
        wins.append((lo, hi))
        cs = [1000, 4096, 7777][i % 3]
        chunks = []
        for s in range(0, len(x), cs):
            part = x[s:s + cs]
            kind = (i + s // cs) % 4
            if kind == 3:
                chunks.append(fast5.RawChunk(s, len(part), fast5.KIND_RAW, part.tobytes()))
                continue
            v = kind % 2
            body = hw.svb_body(part, v, True)
            if kind < 2:
                f = Z.compress(body, [1, 3, 19][i % 3])
                chunks.append(fast5.RawChunk(s, len(part), v + fast5.KIND_VBZ0_ZSTD, f, True, len(part), len(body)))
            else:
                chunks.append(fast5.RawChunk(s, len(part), v, body, True, len(part)))
        stored.append(fast5.CompressedRead('synthetic', str(i), len(x), chunks))
        hosted.append(fast5.CompressedRead('synthetic', str(i), len(x), [c.unzstd() for c in chunks]))
    return locus, reads, stored, hosted, wins


def _engine(locus):
    from warpstr_b200.automata import StateAutomata
    from warpstr_b200.caller import CallerEngine
    eng = CallerEngine()
    ids = [eng.add_automaton(StateAutomata(rx), locus.flank_length) for rx in (locus.template_regex,
                                                                               locus.reverse_regex)]
    return eng, ids


def test_call_arrays_vbz_from_frames_matches_bodies(built_lib):
    from warpstr_b200.caller import pack_vbz
    locus, reads, stored, hosted, wins = _mixed_reads(1500, 51)
    eng, ids = _engine(locus)
    aut = np.array([ids[int(r.reverse)] for r in reads], dtype=np.int32)
    rev = np.array([r.reverse for r in reads], dtype=np.uint8)
    lo, hi = [w[0] for w in wins], [w[1] for w in wins]
    res = []
    for comp in (hosted, stored):
        host, table, read_chunk, raw_off = pack_vbz(comp)
        r = eng.call_arrays_vbz(host, table, read_chunk, raw_off, lo, hi, aut, rev, 'Brute', chunk_reads=600)
        res.append({k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in r.items()})
    a, b = res
    host, table, _, _ = pack_vbz(stored)
    assert (table['zstd_off'] >= 0).sum() > 1000 and int(host.numel()) < int(pack_vbz(hosted)[0].numel())
    assert not b['chunk_status'].any() and not b['zstd_status'].any() and not a['zstd_status'].any()
    assert (a['status'] == 0).mean() > 0.9
    for k in ('len1', 'len2', 'status', 'ttest_ties', 'lengths', 'shift_scale'):
        assert np.array_equal(a[k], b[k]), k
    for k in ('cost1', 'cost2'):
        assert np.array_equal(a[k].view(np.int64), b[k].view(np.int64)), k
    for r in range(len(reads)):
        s0 = int(a['seq_off'][r])
        for k, ln in (('seq1', 'len1'), ('seq2', 'len2')):
            assert np.array_equal(a[k][s0:s0 + max(a[ln][r], 0)], b[k][s0:s0 + max(b[ln][r], 0)]), (r, k)


def test_locate_from_frames_matches_bodies(built_lib):
    from warpstr_b200.caller import pack_vbz
    locus, reads, stored, hosted, _ = _mixed_reads(300, 61)
    eng, ids = _engine(locus)
    aut = [tuple(ids)] * len(reads)
    a, b = (eng.locate_arrays_vbz(*pack_vbz(comp), aut) for comp in (hosted, stored))
    assert not b['zstd_status'].any() and not b['chunk_status'].any()
    for k, v in a.items():
        if k not in ('chunk_status', 'zstd_status'):
            assert np.array_equal(np.asarray(v), np.asarray(b[k]), equal_nan=True), k


def _files(tmp_path, monkeypatch, filt, level, checksum=False, n_reads=40):
    from test_gpu_vbz import _caller_only_locus
    monkeypatch.setattr(hw, 'zstd_compress', lambda body, lv=1: Z.compress(body, level, checksum=checksum))
    return _caller_only_locus(tmp_path, filt, n_reads=n_reads)


OUTPUTS = ('overview.csv', 'predictions/sequences/all.fasta', 'predictions/sequences/sequences_template.fasta',
           'predictions/sequences/sequences_reverse.fasta')


@pytest.mark.parametrize('filt,level,checksum', [('vbz0', 1, False), ('vbz1', 1, False), ('vbz0', -5, False),
                                                 ('vbz1', 19, False), ('vbz1', 3, True)])
def test_main_wrapper_files_match_host_zstd_route(built_lib, tmp_path, monkeypatch, filt, level, checksum):
    import glob
    import shutil
    from test_gpu_vbz import _run_main
    locus, d = _files(tmp_path, monkeypatch, filt, level, checksum)
    kinds = {c.kind for p in glob.glob(str(tmp_path / '*.fast5')) for rid in fast5.read_names(p)
             for c in fast5.stored_chunks(p, rid).chunks}
    assert kinds == ({0, 1} & {int(filt[3])} if checksum else {int(filt[3]) + fast5.KIND_VBZ0_ZSTD})
    pristine = str(tmp_path / 'pristine.csv')
    shutil.copy(os.path.join(d, 'overview.csv'), pristine)
    _run_main(d, locus)                                             # frames decoded on the device
    got = {f: open(os.path.join(d, f), 'rb').read() for f in OUTPUTS}
    got.update({p: open(p, 'rb').read() for p in glob.glob(os.path.join(d, 'predictions', '**', '*'), recursive=True)
                if os.path.isfile(p)})
    shutil.rmtree(os.path.join(d, 'predictions'))
    shutil.copy(pristine, os.path.join(d, 'overview.csv'))
    stored = fast5.stored_chunks

    def host_zstd(path, read_name=None, h5=None):                  # zstd undone on the host
        r = stored(path, read_name, h5)
        r.chunks = [c.unzstd() for c in r.chunks]
        return r
    monkeypatch.setattr(fast5, 'stored_chunks', host_zstd)
    _run_main(d, locus)
    for f, data in got.items():
        assert open(os.path.join(d, f) if not os.path.isabs(f) else f, 'rb').read() == data, f


def test_main_wrapper_corrupt_frame_raises_naming_the_read(built_lib, tmp_path, monkeypatch):
    from test_gpu_vbz import _run_main
    locus, d = _files(tmp_path, monkeypatch, 'vbz0', 1, n_reads=12)
    path = str(tmp_path / 'batch1.fast5')
    with fast5.H5File(path) as h5:
        obj = h5._object(h5._resolve('read_0001-read/Raw/Signal'))
        _, csize, _, addr = sorted(h5._chunk_entries(obj))[1]
        data = bytes(h5.buf[addr + h5.base:addr + h5.base + csize])
    frame = bytearray(data[4:])
    frame[-1] = 0                                                    # the last bitstream loses its end mark
    n = struct.unpack_from('<I', data, 0)[0] // 2
    assert fast5.zstd_frame_size(bytes(frame), n * 5 + 16) > 0
    assert Z.reference(bytes(frame), fast5.zstd_frame_size(bytes(frame), n * 5 + 16)) is None
    with open(path, 'r+b') as fh:
        fh.seek(addr + 4 + len(frame) - 1)
        fh.write(b'\0')
    before = open(os.path.join(d, 'overview.csv'), 'rb').read()
    with pytest.raises(fast5.Fast5FormatError, match='batch1.fast5: read 0001-read: zstd: corrupt VBZ chunk'):
        _run_main(d, locus)
    assert open(os.path.join(d, 'overview.csv'), 'rb').read() == before
    assert not os.path.exists(os.path.join(d, 'predictions'))
