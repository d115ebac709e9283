"""GPU: VBZ decoding on the device (wstr_vbz_decode_batch) against the host decoder (fast5.vbz_decompress), and
the fast5 route of the caller that uses it (fast5.raw_chunks -> CallerEngine.call_vbz_batch / call_arrays_vbz,
wrapper.main_wrapper)."""
import os

import numpy as np
import pytest

import _h5write as hw
from warpstr_b200 import fast5, synth

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), 'golden')


def _signal(rng, n, wide=False):
    x = (450 + np.cumsum(rng.integers(-60, 61, size=n))).astype(np.int16)
    if wide and n > 20:
        x[3], x[4], x[5] = 32767, -32768, 32767          # +-65535 jumps: 3-byte zig-zag codes in v0
        x[10:14] = (-32768, 32767, 0, -32767)
    return x


def _decode_on_device(chunks, status_init=-7):
    """[(body, n coded, n written, kind, zigzag)] -> (int16 samples of every chunk, status per chunk), one call."""
    import torch
    from warpstr_b200 import _lib
    m = len(chunks)
    in_bytes = np.array([len(c[0]) for c in chunks], dtype=np.int64)
    in_off = np.zeros(m, dtype=np.int64)
    in_off[1:] = np.cumsum((in_bytes[:-1] + 15) & ~15)
    total = int(in_off[-1] + ((in_bytes[-1] + 15) & ~15)) if m else 0
    pay = np.zeros(max(total, 16), dtype=np.uint8)
    for c, o in zip(chunks, in_off):
        pay[o:o + len(c[0])] = np.frombuffer(c[0], dtype=np.uint8)
    n_out = np.array([c[2] for c in chunks], dtype=np.int32)
    out_off = np.zeros(m, dtype=np.int64)
    out_off[1:] = np.cumsum(n_out[:-1].astype(np.int64) + 3)           # odd gaps: every destination alignment
    d_raw = torch.full((int(out_off[-1] + n_out[-1]) + 8 if m else 8,), 12345, dtype=torch.int16, device='cuda')
    d_status = torch.full((max(m, 1),), status_init, dtype=torch.int32, device='cuda')
    ws = torch.empty(_lib.vbz_workspace_bytes(m), dtype=torch.uint8, device='cuda')
    _lib.vbz_decode_batch(torch.from_numpy(pay).cuda(), in_off, in_bytes, [c[1] for c in chunks], n_out,
                          [c[3] for c in chunks], [int(c[4]) for c in chunks], out_off, d_raw, d_status, ws)
    raw = d_raw.cpu().numpy()
    outs = [raw[o:o + k] for o, k in zip(out_off, n_out)]
    gaps = [raw[o + k:o + k + 3] for o, k in zip(out_off, n_out)]
    assert all((g == 12345).all() for g in gaps), 'a chunk wrote outside its output range'
    return outs, d_status.cpu().numpy()[:m]


def _host(body, n, kind, zigzag):
    return np.frombuffer(fast5.vbz_decode_body(body, n, kind, 2, int(zigzag)), dtype='<i2')


@pytest.mark.parametrize('version', [0, 1])
@pytest.mark.parametrize('zigzag', [True, False])
def test_kernel_matches_host_decoder(built_lib, version, zigzag):
    rng = np.random.default_rng(10 * version + zigzag)
    sizes = [0, 1, 3, 4, 5, 8, 9, 1000, 4097, 150000, 1000003]
    chunks, want = [], []
    for n in sizes:
        x = _signal(rng, n, wide=True)
        body = hw.svb_body(x, version, zigzag)
        # the path the host takes: vbz_decompress on the whole stored chunk
        host = np.frombuffer(fast5.vbz_decompress(hw.vbz_chunk(x, version, zstd=True, zigzag=zigzag),
                                                  (version, 2, int(zigzag), 1)), dtype='<i2')
        assert np.array_equal(host, x)
        chunks.append((body, n, n, version, zigzag))
        want.append(host)
    got, status = _decode_on_device(chunks)
    assert not status.any()
    for n, g, w in zip(sizes, got, want):
        assert np.array_equal(g, w), n


def test_kernel_wraps_like_numpy(built_lib):
    """Bodies no 16-bit encoder writes -- v0 deltas far outside int16 -- still decode as numpy's int64 cumsum
    cast to int16; and a chunk coding more samples than it writes (HDF5's last chunk)."""
    rng = np.random.default_rng(3)
    n = 5000
    zz = rng.integers(0, 2 ** 32, size=n, dtype=np.uint64)
    nb = 1 + (zz >= 1 << 8) + (zz >= 1 << 16) + (zz >= 1 << 24)
    codes = np.zeros((n + 3) // 4 * 4, dtype=np.uint8)
    codes[:n] = nb - 1
    ctrl = (codes.reshape(-1, 4) << np.array([0, 2, 4, 6], dtype=np.uint8)).sum(axis=1).astype(np.uint8)
    data = zz.astype('<u4').view(np.uint8).reshape(n, 4)[np.arange(4)[None, :] < nb[:, None]]
    body = ctrl.tobytes() + data.tobytes() + b'\x01\x02\x03'                 # v0 allows trailing bytes
    chunks = [(body, n, n, 0, True), (body, n, n, 0, False), (body, n, 1234, 0, True)]
    got, status = _decode_on_device(chunks)
    assert not status.any()
    assert np.array_equal(got[0], _host(body, n, 0, True))
    assert np.array_equal(got[1], _host(body, n, 0, False))
    assert np.array_equal(got[2], _host(body, n, 0, True)[:1234])


def test_many_mixed_chunks(built_lib):
    rng = np.random.default_rng(7)
    chunks, want = [], []
    for i in range(5200):
        n = int(rng.choice([0, 1, 2, 7, 33, 100, 4095, 4096, 4097, 9000, int(rng.integers(0, 20000))]))
        x = _signal(rng, n, wide=bool(i % 3 == 0))
        kind = int(rng.integers(0, 3))
        zigzag = bool(rng.integers(0, 2)) if kind != 2 else False
        if kind == 2:
            chunks.append((x.tobytes(), n, n, 2, False))
            want.append(x)
        else:
            body = hw.svb_body(x, kind, zigzag)
            keep = int(rng.integers(0, n + 1)) if i % 5 == 0 else n
            chunks.append((body, n, keep, kind, zigzag))
            want.append(_host(body, n, kind, zigzag)[:keep])
    got, status = _decode_on_device(chunks)
    assert not status.any()
    for i, (g, w) in enumerate(zip(got, want)):
        assert np.array_equal(g, w), i


def test_bad_chunks_get_the_host_error_and_spare_their_neighbours(built_lib):
    rng = np.random.default_rng(11)
    x = _signal(rng, 3000, wide=True)
    good0, good1 = hw.svb_body(x, 0, True), hw.svb_body(x, 1, True)
    n_ctrl0, n_key1 = (3000 + 3) // 4, (3000 + 7) // 8
    cases = [
        (good0[:n_ctrl0 - 1], 1),                    # truncated control block
        (good0[:-1], 2),                             # v0 data shorter than the codes need
        (good1[:n_key1 - 3], 1),                     # truncated key block
        (good1[:-1], 3),                             # v1 data one byte short
        (good1 + b'\x00', 3),                        # v1 data one byte long
    ]
    kinds = [0, 0, 1, 1, 1]
    table, want_status = [], []
    for (body, st), kind in zip(cases, kinds):
        table.append((good0 if kind == 0 else good1, 3000, 3000, kind, True))
        want_status.append(0)
        table.append((body, 3000, 3000, kind, True))
        want_status.append(st)
        with pytest.raises(fast5.Fast5FormatError):                   # the host refuses the same chunk
            fast5.vbz_decode_body(body, 3000, kind, 2, 1)
    table.append((good1, 3000, 3000, 1, True))
    want_status.append(0)
    got, status = _decode_on_device(table)
    assert status.tolist() == want_status
    for i, st in enumerate(want_status):
        if st == 0:
            assert np.array_equal(got[i], x), i


# -- the caller on compressed reads -------------------------------------------------------------------------
def _c1():
    z = np.load(os.path.join(GOLD, 'c1_bundled.npz'))
    raws = [np.cumsum(z[f'raw_delta{i}'].astype(np.int64)).astype(np.int16) for i in range(len(z['names']))]
    wins = list(zip(z['l_start_raw'].tolist(), z['r_end_raw'].tolist()))
    return z, raws, wins


@pytest.mark.parametrize('filt', ['vbz0', 'vbz1'])
@pytest.mark.parametrize('chunk', [4000, 102400])
def test_bundled_reads_compressed(built_lib, tmp_path, filt, chunk):
    from warpstr_b200.wrapper import CallerWrapper, Locus, flanks_from_template
    z, raws, wins = _c1()
    path = str(tmp_path / 'c1.fast5')
    names = [str(n) for n in z['names']]
    hw.write_multi(path, dict(zip(names, raws)), filt, chunk=chunk)
    reads = [fast5.raw_chunks(path, nm) for nm in names]
    assert all(np.array_equal(r.decode(), x) for r, x in zip(reads, raws))
    locus = Locus(name='Human_STR_1108232', sequence=str(z['sequence']), flank_length=int(z['flank_length']))
    cw = CallerWrapper(locus, threads=2, flanks=flanks_from_template(str(z['left']), str(z['right'])))
    rev = [bool(r) for r in z['reverse']]
    res = cw.run_compressed(reads, wins, rev)
    assert [r.resc_seq for r in res] == [str(s) for s in z['resc_seq']]
    assert [r.seq for r in res] == [str(s) for s in z['seq']]
    assert [r.cost for r in res] == z['cost1'].tolist()
    assert [r.resc_cost for r in res] == z['cost2'].tolist()
    assert sorted(set(len(r.resc_seq) for r in res)) == [40, 44]
    assert res == cw.run_raw(raws, wins, rev)


def test_synthetic_batch_matches_raw_route(built_lib):
    import torch
    from warpstr_b200.automata import StateAutomata
    from warpstr_b200.caller import CallerEngine, pack_vbz
    locus = synth.make_locus('HD', seed=31)
    stas = [StateAutomata(locus.template_regex), StateAutomata(locus.reverse_regex)]
    reads = synth.make_reads(locus, 2000, seed=32, noise=0.2)
    eng = CallerEngine()
    ids = [eng.add_automaton(s, locus.flank_length) for s in stas]
    rng = np.random.default_rng(33)
    raws, wins = [], []
    for r in reads:
        raw, lo, hi = synth.to_raw_int16(rng, r.signal, pad=int(rng.integers(100, 3000)), spike_rate=5e-4)
        raws.append(raw)
        wins.append((lo, hi))
    aut = np.array([ids[int(r.reverse)] for r in reads], dtype=np.int32)
    rev = np.array([r.reverse for r in reads], dtype=np.uint8)
    comp = []
    for i, x in enumerate(raws):                       # chunk sizes and VBZ versions vary from read to read
        cs = [1000, 4096, 7777][i % 3]
        chunks = []
        for s in range(0, len(x), cs):
            part = x[s:s + cs]
            kind = (i + s // cs) % 3
            if kind == 2:
                chunks.append(fast5.RawChunk(s, len(part), 2, part.tobytes()))
            else:
                chunks.append(fast5.RawChunk(s, len(part), kind, hw.svb_body(part, kind, True), True, len(part)))
        comp.append(fast5.CompressedRead('synthetic', str(i), len(x), chunks))
    roff = np.zeros(len(raws) + 1, dtype=np.int64)
    roff[1:] = np.cumsum([len(x) for x in raws])
    lo, hi = [w[0] for w in wins], [w[1] for w in wins]
    a = eng.call_arrays_raw(torch.from_numpy(np.concatenate(raws)).pin_memory(), roff, lo, hi, aut, rev, 'Brute')
    a = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in a.items()}
    host, table, read_chunk, raw_off = pack_vbz(comp)
    assert np.array_equal(raw_off, roff)
    b = eng.call_arrays_vbz(host, table, read_chunk, raw_off, lo, hi, aut, rev, 'Brute')
    assert not b['chunk_status'].any()
    assert (a['status'] == 0).mean() > 0.9
    for k in ('len1', 'len2', 'status', 'ttest_ties', 'lengths', 'shift_scale'):
        assert np.array_equal(a[k], b[k]), k
    for k in ('cost1', 'cost2'):
        assert np.array_equal(a[k].view(np.int64), b[k].view(np.int64)), k
    for r in range(len(reads)):
        s0 = int(a['seq_off'][r])
        for k, ln in (('seq1', 'len1'), ('seq2', 'len2')):
            assert np.array_equal(a[k][s0:s0 + max(a[ln][r], 0)], b[k][s0:s0 + max(b[ln][r], 0)]), (r, k)


def _caller_only_locus(tmp_path, filt, n_reads=40, files=3, corrupt=False):
    """Multi-read files written with the test writer, a caller_only overview of their reads."""
    from warpstr_b200 import caller_only
    locus = synth.make_locus('HD', seed=41)
    reads = synth.make_reads(locus, n_reads, seed=42, noise=0.2)
    rng = np.random.default_rng(43)
    rows = []
    per_file = [dict() for _ in range(files)]
    for i, r in enumerate(reads):
        raw, lo, hi = synth.to_raw_int16(rng, r.signal, pad=2000, spike_rate=5e-4)
        rid = f'{i:04d}-read'
        per_file[i % files][rid] = raw
        rows.append((i % files, rid, r.reverse, lo, hi))
    paths = []
    for k, d in enumerate(per_file):
        p = str(tmp_path / f'batch{k}.fast5')
        hw.write_multi(p, d, filt, chunk=3000, root='symtab' if k % 2 == 0 else 'links')
        paths.append(p)
    if corrupt:
        hw.corrupt_vbz_chunk(paths[1], rows[1][1], 1)
    csv_path = str(tmp_path / 'reads.csv')
    with open(csv_path, 'w') as fh:
        fh.write('fast5_path,locus,read_name,reverse,l_start_raw,r_end_raw\n')
        for k, rid, rv, lo, hi in rows:
            fh.write(f'{paths[k]},LOC,{rid},{rv},{lo},{hi}\n')
    out = str(tmp_path / 'out')
    caller_only.prepare(out, csv_path)
    return locus, os.path.join(out, 'LOC')


def _run_main(locus_dir, locus, workload=None):
    from warpstr_b200.wrapper import Locus, flanks_from_template, main_wrapper
    loc = Locus(name='LOC', sequence=locus.sequence, flank_length=locus.flank_length, path=locus_dir)
    return main_wrapper(loc, workload=workload, flanks=flanks_from_template(locus.left, locus.right))


@pytest.mark.parametrize('filt', ['vbz0', 'vbz1-raw'])
def test_main_wrapper_files_byte_identical(built_lib, tmp_path, filt):
    import shutil
    from warpstr_b200.overview import load_overview
    from warpstr_b200.wrapper import get_workload
    locus, d = _caller_only_locus(tmp_path, filt)
    pristine = os.path.join(str(tmp_path), 'pristine.csv')
    shutil.copy(os.path.join(d, 'overview.csv'), pristine)
    _run_main(d, locus)                                          # the file route: device decode
    got = {f: open(os.path.join(d, f), 'rb').read() for f in ('overview.csv', 'predictions/sequences/all.fasta',
                                                              'predictions/sequences/sequences_template.fasta',
                                                              'predictions/sequences/sequences_reverse.fasta')}
    shutil.rmtree(os.path.join(d, 'predictions'))
    shutil.copy(pristine, os.path.join(d, 'overview.csv'))
    _, df = load_overview(d)
    _run_main(d, locus, workload=get_workload(df, d))            # host decode, float64 windows
    for f, data in got.items():
        assert open(os.path.join(d, f), 'rb').read() == data, f


def test_main_wrapper_corrupt_chunk_raises_and_writes_nothing(built_lib, tmp_path):
    locus, d = _caller_only_locus(tmp_path, 'vbz0-raw', n_reads=12, corrupt=True)
    before = open(os.path.join(d, 'overview.csv'), 'rb').read()
    with pytest.raises(fast5.Fast5FormatError, match='0001-read'):
        _run_main(d, locus)
    assert open(os.path.join(d, 'overview.csv'), 'rb').read() == before
    assert not os.path.exists(os.path.join(d, 'predictions'))
