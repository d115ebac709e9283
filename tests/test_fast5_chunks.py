"""CPU: the fast5 reader on files written by tests/_h5write.py -- every layout and filter it parses -- and the
chunk form of a read's signal the device decoder takes (fast5.raw_chunks, wrapper.get_compressed_workload)."""
import os

import numpy as np
import pytest

import _h5write as hw
from warpstr_b200 import fast5

FILTERS = ['vbz0', 'vbz1', 'vbz0-raw', 'vbz1-raw', 'vbz0-nozz', 'deflate', 'none', 'contiguous']
KINDS = {'vbz0': {0}, 'vbz1': {1}, 'vbz0-raw': {0}, 'vbz1-raw': {1}, 'vbz0-nozz': {0}, 'deflate': {2}, 'none': {2},
         'contiguous': {2}}


def _reads(seed=0):
    rng = np.random.default_rng(seed)
    out = {}
    for i, n in enumerate([1, 999, 1000, 4097, 10001]):
        x = (450 + np.cumsum(rng.integers(-50, 51, size=n))).astype(np.int16)
        if n > 10:
            x[5], x[6], x[7] = 32767, -32768, 32767
        out[f'{i:02d}ab-cd'] = x
    return out


@pytest.mark.parametrize('filt', FILTERS)
@pytest.mark.parametrize('root', ['symtab', 'links'])
def test_multi_read_files(tmp_path, filt, root):
    reads = _reads()
    p = str(tmp_path / 'm.fast5')
    hw.write_multi(p, reads, filt, chunk=1000, root=root, fanout=2)
    assert fast5.read_names(p) == sorted(reads)
    for rid, x in reads.items():
        got = fast5.raw_signal(p, rid)
        assert got.dtype == np.int16 and np.array_equal(got, x)
        assert np.array_equal(fast5.raw_signal(p, 'read_' + rid), x)
        cr = fast5.raw_chunks(p, rid)
        assert cr.n_samples == len(x) and cr.path == p and cr.read_name == rid
        assert np.array_equal(cr.decode(), got)
        assert {c.kind for c in cr.chunks} == KINDS[filt]
        starts = [c.start for c in cr.chunks]
        assert starts == sorted(starts) and sum(c.count for c in cr.chunks) == len(x)
        for c in cr.chunks:
            if c.kind != fast5.KIND_RAW:
                assert c.zigzag == (filt != 'vbz0-nozz') and c.coded == 1000        # the last chunk is coded whole
                assert np.array_equal(c.decode(), x[c.start:c.start + c.count])


@pytest.mark.parametrize('filt', ['vbz0', 'vbz1', 'deflate', 'contiguous'])
def test_single_read_files(tmp_path, filt):
    x = _reads()['03ab-cd']
    for root in ('symtab', 'links'):
        p = str(tmp_path / f'{root}.fast5')
        hw.write_single(p, x, read_number=12, filt=filt, chunk=700, root=root)
        assert np.array_equal(fast5.raw_signal(p), x)
        # a single-read file has one read, whatever name is asked for (schemas/fast5.py:50-52)
        assert np.array_equal(fast5.raw_signal(p, 'other'), x)
        for name in (None, 'other'):
            cr = fast5.raw_chunks(p, name)
            assert np.array_equal(cr.decode(), x) and {c.kind for c in cr.chunks} == KINDS[filt]


def test_read_selection_matches_raw_signal(tmp_path):
    reads = _reads()
    p = str(tmp_path / 'm.fast5')
    hw.write_multi(p, reads, 'vbz0')
    with pytest.raises(KeyError):
        fast5.raw_signal(p, 'nope')
    with pytest.raises(KeyError):
        fast5.raw_chunks(p, 'nope')
    with pytest.raises(KeyError):          # several reads and no name
        fast5.raw_signal(p)
    with pytest.raises(KeyError):
        fast5.raw_chunks(p)
    one = str(tmp_path / 'one.fast5')
    hw.write_multi(one, {'only': reads['02ab-cd']}, 'vbz1')
    assert np.array_equal(fast5.raw_signal(one), reads['02ab-cd'])
    assert np.array_equal(fast5.raw_chunks(one).decode(), reads['02ab-cd'])


def test_damaged_chunk(tmp_path):
    """A chunk whose codes need more data than it holds: the host decoder refuses it; raw_chunks leaves it
    to the device decoder, whose status says the same (tests/test_gpu_vbz.py)."""
    reads = _reads()
    p = str(tmp_path / 'm.fast5')
    hw.write_multi(p, reads, 'vbz0-raw', chunk=1000)
    hw.corrupt_vbz_chunk(p, '04ab-cd', 2)
    with pytest.raises(fast5.Fast5FormatError):
        fast5.raw_signal(p, '04ab-cd')
    cr = fast5.raw_chunks(p, '04ab-cd')
    with pytest.raises(fast5.Fast5FormatError):
        cr.decode()
    assert np.array_equal(fast5.raw_chunks(p, '03ab-cd').decode(), reads['03ab-cd'])


def _caller_only_overview(tmp_path, with_annot=False):
    from warpstr_b200 import caller_only
    reads = _reads(5)
    names = sorted(reads)
    files = [str(tmp_path / 'a.fast5'), str(tmp_path / 'b.fast5')]
    hw.write_multi(files[0], {k: reads[k] for k in names[:3]}, 'vbz0')
    hw.write_multi(files[1], {k: reads[k] for k in names[3:]}, 'vbz1', root='links')
    csv_path = str(tmp_path / 'reads.csv')
    with open(csv_path, 'w') as fh:
        fh.write('fast5_path,locus,read_name,reverse,l_start_raw,r_end_raw\n')
        for i, k in enumerate(names):
            fh.write(f'{files[0] if i < 3 else files[1]},LOC,{k},{i % 2 == 1},{i},{i + 500}\n')
    out = str(tmp_path / 'out')
    caller_only.prepare(out, csv_path)
    d = os.path.join(out, 'LOC')
    if with_annot:       # an annotated single-read file takes precedence over the row's fast5_path
        annot = os.path.join(d, 'fast5', 'run_0', 'annot')
        os.makedirs(annot)
        hw.write_single(os.path.join(annot, names[1] + '.fast5'), reads[names[0]], filt='vbz1')
    return reads, files, d


@pytest.mark.parametrize('with_annot', [False, True])
def test_compressed_workload_matches_raw_workload(tmp_path, monkeypatch, with_annot):
    from warpstr_b200.overview import load_overview
    from warpstr_b200.wrapper import get_compressed_workload, get_raw_workload
    reads, files, d = _caller_only_overview(tmp_path, with_annot)
    _, df = load_overview(d)
    want = get_raw_workload(df, d)
    opened = []
    real = fast5.H5File.__init__

    def counting(self, path):
        opened.append(path)
        real(self, path)
    monkeypatch.setattr(fast5.H5File, '__init__', counting)
    names, revs, comp, wins = get_compressed_workload(df, d)
    assert sorted(opened) == sorted(set(opened))            # every file parsed once
    assert set(files) <= set(opened)
    assert names == want[0] and revs == want[1] and wins == want[3]
    for r, x in zip(comp, want[2]):
        assert np.array_equal(r.decode(), x)
    assert with_annot == np.array_equal(comp[1].decode(), reads[names[0]])
