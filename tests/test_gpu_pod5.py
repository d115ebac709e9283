"""GPU: reads from POD5 files through the device chain (zstd -> StreamVByte -> normalisation -> window search and
strand detection -> both DP passes) give what the same reads give from fast5 files: main_wrapper's files byte
for byte, CallerEngine.call_vbz_batch / locate_compressed result for result, and a corrupted frame the same
error path."""
import os

import numpy as np
import pytest

import _h5write as hw
import _pod5write as pw
import _zstd as Z
from warpstr_b200 import fast5, pod5, synth

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), 'golden')


def _fixture():
    z = np.load(os.path.join(GOLD, 'c1_bundled.npz'))
    raws = [np.cumsum(z[f'raw_delta{i}'].astype(np.int64)).astype(np.int16) for i in range(len(z['names']))]
    return z, [str(n) for n in z['names']], raws


def _bundled_files(tmp_path, z, names, raws):
    """The ten reads in two POD5 files (2 to 4 rows per read, scattered over the signal table) and the same
    split in two fast5 files of the same stem."""
    p5, f5 = [], []
    for k in range(2):
        part = {n: raws[i] for i, n in enumerate(names) if i % 2 == k}
        p = str(tmp_path / f'run{k}.pod5')
        pw.write(p, part, rows=lambda i, n: 2 + i % 3, seed=k, shuffle=True, signal_batch=5)
        p5.append(p)
        f = str(tmp_path / f'run{k}.fast5')
        hw.write_multi(f, part, 'vbz1', chunk=4000)
        f5.append(f)
    return p5, f5


def test_bundled_reads_from_pod5(built_lib, tmp_path):
    from test_gpu_strand import _bundled_locus, _main_wrapper
    from warpstr_b200.wrapper import CallerWrapper, Locus, flanks_from_template
    z, names, raws = _fixture()
    p5, f5 = _bundled_files(tmp_path, z, names, raws)
    reads = [fast5.stored_chunks(p5[i % 2], n) for i, n in enumerate(names)]
    assert all(len(r.chunks) >= 2 and {c.kind for c in r.chunks} == {fast5.KIND_VBZ1_ZSTD} for r in reads)
    assert all(np.array_equal(r.decode(), x) for r, x in zip(reads, raws))
    locus = Locus(name='Human_STR_1108232', sequence=str(z['sequence']), flank_length=int(z['flank_length']))
    cw = CallerWrapper(locus, threads=2, flanks=flanks_from_template(str(z['left']), str(z['right'])))
    wins = list(zip(z['l_start_raw'].tolist(), z['r_end_raw'].tolist()))
    res = cw.run_compressed(reads, wins, [bool(r) for r in z['reverse']])
    assert [r.resc_seq for r in res] == [str(s) for s in z['resc_seq']]
    assert [r.seq for r in res] == [str(s) for s in z['seq']]
    assert [r.cost for r in res] == z['cost1'].tolist()
    assert [r.resc_cost for r in res] == z['cost2'].tolist()

    loc = _bundled_locus(z)
    for tag, cells in (('given', lambda i: (bool(z['reverse'][i]), int(z['l_start_raw'][i]), int(z['r_end_raw'][i]))),
                       ('located', lambda i: ('', '', ''))):
        out = {}
        for kind, paths in (('pod5', p5), ('fast5', f5)):
            out[kind] = _main_wrapper(tmp_path, f'{tag}_{kind}', loc,
                                      [(paths[i % 2], n) + cells(i) for i, n in enumerate(names)])
        (df, files), (_, files5) = out['pod5'], out['fast5']
        df = df.loc[names]
        assert df['results'].tolist() == z['len2'].tolist() and df['orig'].tolist() == z['len1'].tolist()
        assert sorted(set(df['results'])) == [40, 44]
        assert df['reverse'].tolist() == [bool(r) for r in z['reverse']]
        if tag == 'given':
            np.testing.assert_allclose(df['dtw_cost1'], z['cost1'], rtol=1e-12)
            np.testing.assert_allclose(df['dtw_cost2'], z['cost2'], rtol=1e-12)
        assert set(files) == set(files5) and 'overview.csv' in files
        for f, data in files.items():                      # the only difference: the source column's paths
            assert data.replace(b'.pod5', b'.fast5') == files5[f], (tag, f)


def _locus_files(tmp_path, n_reads=40, files=3):
    """A synthetic HD locus: the reads in ``files`` POD5 files (1 to 3 rows a read) and in as many fast5 files."""
    import uuid
    locus = synth.make_locus('HD', seed=41)
    reads = synth.make_reads(locus, n_reads, seed=42, noise=0.2)
    rng = np.random.default_rng(43)
    per_file = [dict() for _ in range(files)]
    rows = []
    for i, r in enumerate(reads):
        raw, lo, hi = synth.to_raw_int16(rng, r.signal, pad=2000, spike_rate=5e-4)
        rid = str(uuid.UUID(bytes=rng.bytes(16)))
        per_file[i % files][rid] = raw
        rows.append((i % files, rid, r.reverse, lo, hi))
    p5, f5 = [], []
    for k, d in enumerate(per_file):
        p5.append(str(tmp_path / f'batch{k}.pod5'))
        pw.write(p5[-1], d, rows=lambda i, n: 1 + i % 3, seed=k, shuffle=True, signal_batch=7, reads_batch=5)
        f5.append(str(tmp_path / f'batch{k}.fast5'))
        hw.write_multi(f5[-1], d, 'vbz1', chunk=3000)
    return locus, rows, p5, f5


def test_synthetic_locus_pod5_matches_fast5(built_lib, tmp_path):
    from warpstr_b200.caller import CallerResult, pack_vbz
    from warpstr_b200.wrapper import CallerWrapper, Locus, flanks_from_template
    locus, rows, p5, f5 = _locus_files(tmp_path)
    cw = CallerWrapper(Locus(name='LOC', sequence=locus.sequence, flank_length=locus.flank_length), threads=1,
                       flanks=flanks_from_template(locus.left, locus.right))
    wins = [(lo, hi) for _, _, _, lo, hi in rows]
    rev = [bool(rv) for _, _, rv, _, _ in rows]
    got = {}
    for kind, paths in (('pod5', p5), ('fast5', f5)):
        reads = [fast5.stored_chunks(paths[k], rid) for k, rid, _, _, _ in rows]
        if kind == 'pod5':
            assert {c.kind for r in reads for c in r.chunks} == {fast5.KIND_VBZ1_ZSTD}
        eng = cw.engine
        arr = eng.call_arrays_vbz(*pack_vbz(reads), [w[0] for w in wins], [w[1] for w in wins],
                                  np.array(cw._aut(rev), dtype=np.int32), np.array(rev, dtype=np.uint8), 'Brute')
        assert not arr['chunk_status'].any() and not arr['zstd_status'].any(), kind
        got[kind] = (eng.call_vbz_batch(reads, wins, cw._aut(rev), rev, 'Brute'),
                     cw.locate_compressed(reads, [None] * len(reads)))
    (calls, loc), (calls5, loc5) = got['pod5'], got['fast5']
    assert calls == calls5
    assert all(isinstance(c, CallerResult) for c in calls)
    assert set(loc) == set(loc5)
    for k in loc:
        assert np.array_equal(np.asarray(loc[k]), np.asarray(loc5[k]), equal_nan=True), k
    assert (loc['status'] == 0).mean() > 0.9


def test_corrupt_pod5_frame_raises_naming_the_read(built_lib, tmp_path):
    from test_gpu_vbz import _run_main
    from warpstr_b200 import caller_only
    locus, rows, p5, _ = _locus_files(tmp_path, n_reads=12)
    victim = rows[1][1]
    with pod5.Pod5File(p5[1]) as f:
        frame = f.read_chunks(victim, True).chunks[0].payload
        n = f.read_chunks(victim, True).chunks[0].count
    bad = bytearray(frame)
    bad[-1] = 0                                                 # the last bitstream loses its end mark
    assert fast5.zstd_frame_size(bytes(bad), 5 * n + 16) > 0
    assert Z.reference(bytes(bad), fast5.zstd_frame_size(bytes(bad), 5 * n + 16)) is None
    data = open(p5[1], 'rb').read()
    at = data.find(frame)
    assert at > 0 and data.find(frame, at + 1) < 0
    with open(p5[1], 'r+b') as fh:
        fh.seek(at + len(frame) - 1)
        fh.write(b'\0')
    csv_path = str(tmp_path / 'reads.csv')
    with open(csv_path, 'w') as fh:
        fh.write('fast5_path,locus,read_name,reverse,l_start_raw,r_end_raw\n')
        for k, rid, rv, lo, hi in rows:
            fh.write(f'{p5[k]},LOC,{rid},{rv},{lo},{hi}\n')
    caller_only.prepare(str(tmp_path / 'out'), csv_path)
    d = str(tmp_path / 'out' / 'LOC')
    before = open(os.path.join(d, 'overview.csv'), 'rb').read()
    with pytest.raises(fast5.Fast5FormatError, match=f'batch1.pod5: read {victim}: zstd: corrupt VBZ chunk'):
        _run_main(d, locus)
    assert open(os.path.join(d, 'overview.csv'), 'rb').read() == before
    assert not os.path.exists(os.path.join(d, 'predictions'))
