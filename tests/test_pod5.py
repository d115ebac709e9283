"""POD5 reader (warpstr_b200/pod5.py) on files from the test writer (_pod5write.py) and, where pyarrow is
installed, on Arrow IPC files pyarrow writes; the container dispatch of fast5.py and caller_only on POD5 sources."""
import io
import os
import subprocess
import sys
import uuid

import numpy as np
import pytest

import _h5write as hw
import _pod5write as pw
import _zstd as Z
from warpstr_b200 import caller_only, fast5, pod5

SIZES = [0, 1, 7, 8, 9, 102400 + 5]


def _reads(seed, sizes=SIZES):
    rng = np.random.default_rng(seed)
    out = {}
    for n in sizes:
        x = rng.integers(-32767, 32768, size=n).astype(np.int16)
        if n > 4:
            x[:4] = (32767, -32767, 32767, -32767)               # the widest deltas, both ways
        out[str(uuid.UUID(bytes=rng.bytes(16)))] = x
    return out


@pytest.mark.parametrize('rows', [1, 2, 3, 4])
@pytest.mark.parametrize('compressed', [True, False])
def test_round_trip(tmp_path, rows, compressed):
    reads = _reads(rows)
    path = str(tmp_path / 'run.pod5')
    pw.write(path, reads, rows=rows, seed=rows, shuffle=rows > 1, signal_batch=5, reads_batch=4,
             compressed=compressed)
    assert pod5.read_names(path) == list(reads) == fast5.read_names(path)
    with pod5.Pod5File(path) as f:
        for rid, x in reads.items():
            sig = pod5.raw_signal(path, rid)
            assert sig.dtype == np.int16 and np.array_equal(sig, x), len(x)
            assert np.array_equal(fast5.raw_signal(path, rid), x)
            for r in (pod5.raw_chunks(path, rid, f), pod5.stored_chunks(path, rid, f), fast5.stored_chunks(path, rid)):
                assert r.read_name == rid and r.path == path and r.n_samples == len(x)
                assert np.array_equal(r.decode(), sig)


def test_chunk_kinds_and_starts(tmp_path):
    reads = _reads(5)
    frames = {}

    def level1_or_checksum(body):                      # every third row's frame carries a content checksum
        f = Z.compress(body, 1, checksum=len(frames) % 3 == 2)
        frames[f] = len(frames) % 3 == 2
        return f
    path = str(tmp_path / 'run.pod5')
    t = pw.write(path, reads, rows=3, seed=5, shuffle=True, compress=level1_or_checksum)
    plain = str(tmp_path / 'plain.pod5')
    pw.write(plain, reads, rows=3, seed=5, shuffle=True, compressed=False)
    for k, (rid, x) in enumerate(reads.items()):
        samples = [t['sig_samples'][r] for r in t['read_rows'][k]]
        starts = np.concatenate(([0], np.cumsum(samples)[:-1])).tolist()
        keep = [(s, n, t['sig_payload'][r]) for s, n, r in zip(starts, samples, t['read_rows'][k]) if n]
        stored = pod5.stored_chunks(path, rid)
        assert [(c.start, c.count, c.coded) for c in stored.chunks] == [(s, n, n) for s, n, _ in keep]
        for c, (_, n, frame) in zip(stored.chunks, keep):
            assert c.zigzag
            if frames[frame]:                          # the device decoder does not take it: undone here
                assert fast5.zstd_frame_size(frame, 5 * n + 16) < 0
                assert c.kind == fast5.KIND_VBZ1 and c.payload == fast5.zstd_decompress(frame, 5 * n + 16)
            else:
                assert c.kind == fast5.KIND_VBZ1_ZSTD and c.payload == frame
                assert c.body_size == fast5.zstd_frame_size(frame, 5 * n + 16) == len(c.unzstd().payload)
        assert {c.kind for c in pod5.raw_chunks(path, rid).chunks} <= {fast5.KIND_VBZ1}
        raw = pod5.stored_chunks(plain, rid)
        assert {c.kind for c in raw.chunks} <= {fast5.KIND_RAW} and np.array_equal(raw.decode(), x)
    assert any(frames.values()) and not all(frames.values())


def test_open_raw_goes_by_the_signature(tmp_path):
    reads = _reads(6, [100, 200])
    p5 = str(tmp_path / 'named_like_a.fast5')
    pw.write(p5, reads)
    h5 = str(tmp_path / 'run.fast5')
    hw.write_multi(h5, reads, 'vbz1')
    with fast5.open_raw(p5) as f:
        assert isinstance(f, pod5.Pod5File)
    with fast5.open_raw(h5) as f:
        assert isinstance(f, fast5.H5File)
    for rid, x in reads.items():
        a, b = fast5.stored_chunks(p5, rid), fast5.stored_chunks(h5, rid)
        assert np.array_equal(a.decode(), b.decode()) and np.array_equal(a.decode(), x)
    assert issubclass(pod5.Pod5FormatError, fast5.Fast5FormatError)


# -- refusals -------------------------------------------------------------------------------------------------
TAMPER = {
    'row out of range': (lambda t: t['read_rows'][1].append(10 ** 6), 'out of range'),
    'row of another read': (lambda t: t['sig_read_ids'].__setitem__(t['read_rows'][2][0], t['read_ids'][3]),
                            'belongs to read'),
    'row used by two reads': (lambda t: t['read_rows'][3].append(t['read_rows'][4][0]), 'used more than once'),
    'samples != num_samples': (lambda t: t['num_samples'].__setitem__(5, t['num_samples'][5] + 1),
                               'num_samples says'),
    'duplicate read ID': (lambda t: t['read_ids'].__setitem__(2, t['read_ids'][1]), 'appears twice'),
}


@pytest.mark.parametrize('case', sorted(TAMPER))
def test_inconsistent_tables_are_refused(tmp_path, case):
    tamper, msg = TAMPER[case]
    path = str(tmp_path / 'bad.pod5')
    pw.write(path, _reads(7), rows=2, shuffle=True, signal_batch=4, tamper=tamper)
    with pytest.raises(pod5.Pod5FormatError, match=msg) as err:
        fast5.read_names(path)
    assert path in str(err.value)


def _bytes_edit(path, edit):
    data = bytearray(open(path, 'rb').read())
    data = edit(data)
    with open(path, 'wb') as fh:
        fh.write(data)


@pytest.mark.parametrize('case', ['missing read', 'bad signature', 'truncated footer', 'footer length',
                                  'compressed body', 'big-endian', 'unsupported type', 'not arrow'])
def test_bad_files_are_refused(tmp_path, case):
    path = str(tmp_path / 'bad.pod5')
    kw = {'compressed body': dict(compressed_body=True), 'big-endian': dict(big_endian=True),
          'unsupported type': dict(more_columns=[('tags', ('other', 17), np.zeros(6))])}.get(case, {})
    reads = _reads(8)
    pw.write(path, reads, **kw)
    if case == 'bad signature':
        _bytes_edit(path, lambda d: d.__setitem__(1, ord('Q')) or d)
    elif case == 'truncated footer':
        _bytes_edit(path, lambda d: d[:-40])
    elif case == 'footer length':
        _bytes_edit(path, lambda d: d[:-32] + (len(d) * 2).to_bytes(8, 'little') + d[-24:])
    elif case == 'not arrow':
        _bytes_edit(path, lambda d: d[:24] + b'ARROW0' + d[30:])
    msg = {'missing read': 'not found', 'bad signature': 'not an HDF5 file', 'truncated footer': 'truncated',
           'footer length': 'footer', 'compressed body': 'BodyCompression', 'big-endian': 'big-endian',
           'unsupported type': 'Arrow type 17', 'not arrow': 'not an Arrow IPC file'}[case]
    # a damaged signature makes the file neither POD5 nor HDF5, so open_raw leaves it to the HDF5 reader's error
    kind = fast5.Fast5FormatError if case == 'bad signature' else pod5.Pod5FormatError
    with pytest.raises(kind, match=msg) as err:
        if case == 'missing read':
            fast5.raw_signal(path, str(uuid.UUID(int=12345)))
        elif case == 'bad signature':
            fast5.read_names(path)
        else:
            pod5.Pod5File(path).close()
    assert path in str(err.value)
    if case == 'bad signature':
        with pytest.raises(pod5.Pod5FormatError, match='bad signature'):
            pod5.read_names(path)


# -- pyarrow as an independent check of the Arrow layer -------------------------------------------------------
def _arrow_tables(pa, reads, rows, compressed, seed):
    """A Signal and a Reads table written by pyarrow (several batches, rows of a read scattered)."""
    rng = np.random.default_rng(seed)
    pieces, owner = [], []
    for k, x in enumerate(reads.values()):
        cuts = sorted(rng.integers(0, len(x) + 1, size=rows - 1).tolist())
        for a, b in zip([0] + cuts, cuts + [len(x)]):
            pieces.append(x[a:b])
            owner.append(k)
    order = rng.permutation(len(pieces))
    where = np.empty(len(pieces), np.int64)
    where[order] = np.arange(len(pieces))
    ids = [uuid.UUID(r).bytes for r in reads]
    sig_type = pa.large_binary() if compressed else pa.large_list(pa.int16())
    sig_vals = [hw.zstd_compress(hw.svb_body(pieces[p], 1)) if compressed else pieces[p].tolist() for p in order]
    signal = pa.table({'read_id': pa.array([ids[owner[p]] for p in order], pa.binary(16)),
                       'signal': pa.array(sig_vals, sig_type),
                       'samples': pa.array([len(pieces[p]) for p in order], pa.uint32())})
    rows_of = [[] for _ in reads]
    for p, k in enumerate(owner):
        rows_of[k].append(int(where[p]))
    n = len(reads)
    table = pa.table({'read_id': pa.array(ids, pa.binary(16)),
                      'signal': pa.array(rows_of, pa.list_(pa.uint64())),
                      'read_number': pa.array(np.arange(n), pa.uint32()),
                      'pore_type': pa.array(['R9.4.1'] * n).dictionary_encode(),
                      'calibration': pa.array([{'offset': -240.0, 'scale': 0.17}] * n,
                                              pa.struct([('offset', pa.float32()), ('scale', pa.float32())])),
                      'end_reason': pa.DictionaryArray.from_arrays(pa.array(np.arange(n) % 2, pa.int16()),
                                                                   pa.array(['unknown', 'signal_positive'])),
                      'median_before': pa.array(rng.random(n), pa.float32()),
                      'num_samples': pa.array([len(x) for x in reads.values()], pa.uint64())})
    return signal, table


def _ipc(pa, table, chunk):
    sink = io.BytesIO()
    with pa.ipc.new_file(sink, table.schema) as w:
        w.write_table(table, max_chunksize=chunk)
    return sink.getvalue()


@pytest.mark.parametrize('compressed', [True, False])
def test_reads_arrow_files_pyarrow_writes(tmp_path, compressed):
    pa = pytest.importorskip('pyarrow')
    import pyarrow.ipc  # noqa: F401
    reads = _reads(9)
    signal, table = _arrow_tables(pa, reads, 3, compressed, 9)
    path = str(tmp_path / 'pa.pod5')
    pw.container(path, {pw.SIGNAL_TABLE: _ipc(pa, signal, 5), pw.READS_TABLE: _ipc(pa, table, 4)})
    assert pod5.read_names(path) == list(reads)
    with pod5.Pod5File(path) as f:
        for rid, x in reads.items():
            assert np.array_equal(f.read_signal(rid), x)
            kinds = {c.kind for c in f.read_chunks(rid, True).chunks}
            assert kinds <= ({fast5.KIND_VBZ1_ZSTD} if compressed else {fast5.KIND_RAW})


def test_pyarrow_reads_what_the_writer_writes(tmp_path):
    pa = pytest.importorskip('pyarrow')
    import pyarrow.ipc  # noqa: F401
    reads = _reads(10)
    t = pw.write(str(tmp_path / 'w.pod5'), reads, rows=3, shuffle=True, signal_batch=4, reads_batch=4)
    sig = pa.ipc.open_file(pa.BufferReader(t['arrow'][pw.SIGNAL_TABLE])).read_all()
    assert sig.column('read_id').to_pylist() == t['sig_read_ids']
    assert sig.column('signal').to_pylist() == t['sig_payload']
    assert sig.column('samples').to_pylist() == t['sig_samples'] and sig.schema.field('samples').type == pa.uint32()
    assert sig.schema.field('read_id').metadata[b'ARROW:extension:name'] == b'minknow.uuid'
    assert sig.schema.field('signal').metadata[b'ARROW:extension:name'] == b'minknow.vbz'
    assert sig.schema.field('signal').type == pa.large_binary()
    rd = pa.ipc.open_file(pa.BufferReader(t['arrow'][pw.READS_TABLE])).read_all()
    assert rd.column('read_id').to_pylist() == t['read_ids']
    assert rd.column('signal').to_pylist() == t['read_rows']
    assert rd.column('num_samples').to_pylist() == [len(x) for x in reads.values()]
    assert rd.column('end_reason').to_pylist()[:3] == ['unknown', 'signal_positive', 'data_service_unblock_mux_change']
    assert rd.column('calibration').to_pylist()[0] == {'offset': -240.0, 'scale': pytest.approx(0.1755)}
    assert rd.schema.field('pore_type').type == pa.dictionary(pa.int16(), pa.string())
    ri = pa.ipc.open_file(pa.BufferReader(t['arrow'][pw.RUN_INFO_TABLE])).read_all()
    assert ri.column('acquisition_id').to_pylist() == ['acq0']
    plain = pw.write(str(tmp_path / 'p.pod5'), reads, rows=2, compressed=False)
    sig = pa.ipc.open_file(pa.BufferReader(plain['arrow'][pw.SIGNAL_TABLE])).read_all()
    assert sig.schema.field('signal').type == pa.large_list(pa.int16())
    assert all(np.array_equal(a, b) for a, b in zip(sig.column('signal').to_pylist(), plain['sig_payload']))


def test_files_without_num_samples_or_run_info(tmp_path):
    reads = _reads(11)
    path = str(tmp_path / 'old.pod5')
    pw.write(path, reads, rows=2, num_samples=False, extra_columns=False, run_info=False)
    for rid, x in reads.items():
        assert np.array_equal(fast5.raw_signal(path, rid), x)


# -- the product does not need pod5 or pyarrow ------------------------------------------------------------------
def test_product_package_does_not_import_pyarrow_or_pod5(tmp_path):
    """pandas imports pyarrow by itself where it is installed, so the route runs with both packages blocked
    (``sys.modules[name] = None`` makes every import of them fail), and no module of the package names them."""
    import ast
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for dirpath, _, files in os.walk(os.path.join(root, 'warpstr_b200')):
        for fn in files:
            if fn.endswith('.py'):
                tree = ast.parse(open(os.path.join(dirpath, fn)).read())
                for node in ast.walk(tree):
                    names = ([a.name for a in node.names] if isinstance(node, ast.Import) else
                             [node.module] if isinstance(node, ast.ImportFrom) and node.level == 0 else [])
                    assert not any(n.split('.')[0] in ('pyarrow', 'pod5', 'lib_pod5') for n in names), (fn, names)
    path = str(tmp_path / 'run.pod5')
    x = _reads(12, [300])
    pw.write(path, x, rows=2)
    code = ("import sys; sys.modules.update(pyarrow=None, pod5=None, lib_pod5=None); "
            "import warpstr_b200.fast5 as f, warpstr_b200.wrapper, warpstr_b200.caller_only; "
            f"print(f.stored_chunks({path!r}, f.read_names({path!r})[0]).decode().tolist())")
    out = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True, cwd=root)
    assert out.returncode == 0 and out.stdout.strip() == str(list(x.values())[0].tolist()), out.stdout + out.stderr


# -- caller_only on POD5 sources ----------------------------------------------------------------------------
def test_caller_only_prepare_on_pod5(tmp_path):
    import pandas as pd
    reads = _reads(13, [500, 600, 700, 800])
    names = list(reads)
    paths = [str(tmp_path / 'a.pod5'), str(tmp_path / 'b.pod5')]
    pw.write(paths[0], {n: reads[n] for n in names[:2]})
    pw.write(paths[1], {n: reads[n] for n in names[2:]}, rows=2)
    csv_path = str(tmp_path / 'reads.csv')
    with open(csv_path, 'w') as fh:
        fh.write('fast5_path,locus,read_name,reverse\n')
        for k, n in enumerate(names):
            fh.write(f'{paths[k // 2]},LOC,{n},{["True", ""][k % 2]}\n')
    written = caller_only.prepare(str(tmp_path / 'out'), csv_path)
    df = pd.read_csv(written['LOC']).set_index('read_name')
    assert df.index.tolist() == names and df['fast5_path'].tolist() == [paths[0]] * 2 + [paths[1]] * 2
    from warpstr_b200.wrapper import get_compressed_workload, get_raw_workload
    got_names, revs, raws, wins = get_raw_workload(df, str(tmp_path / 'out' / 'LOC'))
    assert got_names == names and revs == [True, None] * 2 and wins == [None] * 4
    assert all(np.array_equal(r, reads[n]) for n, r in zip(names, raws))
    _, _, comp, _ = get_compressed_workload(df, str(tmp_path / 'out' / 'LOC'))
    assert all(np.array_equal(c.decode(), reads[n]) for n, c in zip(names, comp))
    with open(csv_path, 'a') as fh:
        fh.write(f'{paths[0]},LOC,{names[3]},True\n')               # a read of the other file
    with pytest.raises(ValueError, match=f'Read {names[3]} not found'):
        caller_only.prepare(str(tmp_path / 'out2'), csv_path)
