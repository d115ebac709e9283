"""Test helper: writes the part of POD5 that warpstr_b200/pod5.py parses, so the reader can be tested without the
pod5 or pyarrow packages.

* A forward flatbuffer builder (tables, strings, vectors of tables and of structs), enough for Arrow's Schema,
  Message and File footers and for POD5's footer (``footer.fbs``).
* A minimal Arrow IPC file writer: schema, dictionary batches, record batches, the file footer.  Types: Int,
  FloatingPoint, Bool, FixedSizeBinary, Binary/LargeBinary/Utf8, List/LargeList, Struct and dictionary-encoded
  columns.  No nulls.
* The POD5 container around the Signal, Reads and Run Info tables; signal rows as POD5 writes them: VBZ version
  1 of 2-byte integers (``_h5write.svb_body(x, 1)``) in one zstd frame per row, or ``large_list<int16>``.
"""
import struct
import uuid
from typing import Callable, Dict, List, Optional, Sequence

import numpy as np

import _h5write as hw

SIGNATURE = b'\x8bPOD\r\n\x1a\n'
READS_TABLE, SIGNAL_TABLE, RUN_INFO_TABLE = 0, 1, 4


# ---------------------------------------------------------------------------------------------------
# flatbuffers
# ---------------------------------------------------------------------------------------------------
class Structs:
    """A vector of structs, each packed with ``fmt`` (8-byte aligned)."""

    def __init__(self, fmt: str, rows: Sequence[tuple]):
        self.fmt, self.rows = fmt, list(rows)


def flatbuffer(root: dict) -> bytes:
    """A table is a dict {field index: ('fmt', scalar) | str | dict (table) | list (of tables) | Structs}.
    Written front to back: a table's vtable just before it, its children after it, so every uoffset points
    forward; scalars are aligned to their size and the whole buffer to 8."""
    buf = bytearray(4)

    def pad(a, extra=0):
        buf.extend(bytes(-(len(buf) + extra) % a))

    def put(obj) -> int:
        if isinstance(obj, (str, bytes)):
            data = obj.encode() if isinstance(obj, str) else obj
            pad(4)
            p = len(buf)
            buf.extend(struct.pack('<I', len(data)) + data + b'\x00')
            return p
        if isinstance(obj, Structs):
            pad(8, 4)
            p = len(buf)
            buf.extend(struct.pack('<I', len(obj.rows)))
            for r in obj.rows:
                buf.extend(struct.pack('<' + obj.fmt, *r))
            return p
        if isinstance(obj, list):
            pad(4)
            p = len(buf)
            buf.extend(struct.pack('<I', len(obj)))
            slots = []
            for _ in obj:
                slots.append(len(buf))
                buf.extend(bytes(4))
            for s, o in zip(slots, obj):
                struct.pack_into('<I', buf, s, put(o) - s)
            return p
        n = max(obj) + 1 if obj else 0
        pad(2)
        vt = len(buf)
        buf.extend(bytes(4 + 2 * n))
        pad(8)
        t = len(buf)
        buf.extend(struct.pack('<i', t - vt))
        offs, children = {}, []
        for i in sorted(obj):
            v = obj[i]
            if isinstance(v, tuple):
                size = struct.calcsize('<' + v[0])
                pad(size)
                offs[i] = len(buf) - t
                buf.extend(struct.pack('<' + v[0], v[1]))
            else:
                pad(4)
                offs[i] = len(buf) - t
                children.append((len(buf), v))
                buf.extend(bytes(4))
        struct.pack_into('<HH', buf, vt, 4 + 2 * n, len(buf) - t)
        for i, o in offs.items():
            struct.pack_into('<H', buf, vt + 4 + 2 * i, o)
        for s, v in children:
            struct.pack_into('<I', buf, s, put(v) - s)
        return t

    struct.pack_into('<I', buf, 0, put(root))
    pad(8)
    return bytes(buf)


# ---------------------------------------------------------------------------------------------------
# Arrow IPC
# ---------------------------------------------------------------------------------------------------
# type specs: ('int', bits, signed) ('float', 32|64) ('bool',) ('fsb', width) ('binary',) ('large_binary',)
# ('utf8',) ('list', child) ('large_list', child) ('struct', [(name, spec)]) ('dict', index_bits, dict_id, values)
# ('other', type id): that type id in the schema, int32 values in the batches (for readers that must refuse it)
_TYPE_ID = dict(int=2, float=3, binary=4, utf8=5, bool=6, list=12, struct=13, fsb=15, large_binary=19, large_list=21)


def _field(name: str, spec, meta: Optional[Dict[str, str]] = None) -> dict:
    kind = spec[0]
    f = {0: name, 1: ('?', True)}
    children = []
    if kind == 'other':                                     # a type id of the caller's choosing, no type fields
        f[2], f[3] = ('B', spec[1]), {}
    elif kind == 'dict':
        f[2], f[3] = ('B', _TYPE_ID['utf8']), {}
        f[4] = {0: ('q', spec[2]), 1: {0: ('i', spec[1]), 1: ('?', True)}, 2: ('?', False)}
    else:
        f[2] = ('B', _TYPE_ID[kind])
        if kind == 'int':
            f[3] = {0: ('i', spec[1]), 1: ('?', spec[2])}
        elif kind == 'float':
            f[3] = {0: ('h', {16: 0, 32: 1, 64: 2}[spec[1]])}
        elif kind == 'fsb':
            f[3] = {0: ('i', spec[1])}
        else:
            f[3] = {}
        if kind in ('list', 'large_list'):
            children = [_field('item', spec[1])]
        elif kind == 'struct':
            children = [_field(n, s) for n, s in spec[1]]
    f[5] = children
    if meta:
        f[6] = [{0: k, 1: v} for k, v in meta.items()]
    return f


def _np_dtype(spec) -> str:
    if spec[0] == 'int':
        return ('<i' if spec[2] else '<u') + str(spec[1] // 8)
    return '<f%d' % (spec[1] // 8)


def _array(spec, data, nodes: list, bufs: list) -> None:
    """Append the field nodes and buffers (bytes) of one column's values ``data`` to ``nodes`` / ``bufs``."""
    kind = spec[0]
    if kind == 'dict':
        kind, spec = 'int', ('int', spec[1], True)
    elif kind == 'other':
        kind, spec = 'int', ('int', 32, True)
    n = len(next(iter(data.values()))) if kind == 'struct' else len(data)
    nodes.append((n, 0))
    bufs.append(b'')                                         # validity: none, no nulls
    if kind in ('int', 'float'):
        bufs.append(np.asarray(data).astype(_np_dtype(spec)).tobytes())
    elif kind == 'bool':
        bufs.append(np.packbits(np.asarray(data, dtype=bool), bitorder='little').tobytes())
    elif kind == 'fsb':
        bufs.append(b''.join(data))
    elif kind in ('binary', 'utf8', 'large_binary'):
        items = [d.encode() if isinstance(d, str) else bytes(d) for d in data]
        offs = np.zeros(n + 1, dtype='<i8' if kind == 'large_binary' else '<i4')
        np.cumsum([len(d) for d in items], out=offs[1:])
        bufs.append(offs.tobytes())
        bufs.append(b''.join(items))
    elif kind in ('list', 'large_list'):
        offs = np.zeros(n + 1, dtype='<i8' if kind == 'large_list' else '<i4')
        np.cumsum([len(d) for d in data], out=offs[1:])
        bufs.append(offs.tobytes())
        child = np.concatenate([np.asarray(d) for d in data]) if n else np.zeros(0)
        _array(spec[1], child, nodes, bufs)
    elif kind == 'struct':
        for (name, s) in spec[1]:
            _array(s, data[name], nodes, bufs)
    else:
        raise ValueError(kind)


def _message(header_type: int, header: dict, body_len: int) -> bytes:
    """An encapsulated message: continuation word, metadata length, the Message flatbuffer padded to 8."""
    fb = flatbuffer({0: ('h', 4), 1: ('B', header_type), 2: header, 3: ('q', body_len)})
    return struct.pack('<Ii', 0xFFFFFFFF, len(fb)) + fb


def _record_batch(spec_cols, length: int, cols: list, compressed: bool = False):
    """(RecordBatch table, body) of one batch."""
    nodes, bufs = [], []
    for spec, data in zip(spec_cols, cols):
        _array(spec, data, nodes, bufs)
    body, layout = bytearray(), []
    for b in bufs:
        layout.append((len(body), len(b)))
        body += b + bytes(-len(b) % 8)
    rb = {0: ('q', length), 1: Structs('qq', nodes), 2: Structs('qq', layout)}
    if compressed:
        rb[3] = {0: ('b', 1), 1: ('b', 0)}                    # ZSTD, per buffer
    return rb, bytes(body)


def arrow_file(columns: list, batches: List[list], schema_meta: Optional[Dict[str, str]] = None,
               compressed_body: bool = False, big_endian: bool = False) -> bytes:
    """An Arrow IPC file.  ``columns``: [(name, spec, field metadata or None)]; ``batches``: per batch, one
    value sequence per column.  Dictionary columns' dictionaries (spec[3], strings) go into dictionary batches."""
    fields = [_field(n, s, m) for n, s, m in columns]
    schema = {0: ('h', int(big_endian)), 1: fields}
    if schema_meta:
        schema[2] = [{0: k, 1: v} for k, v in schema_meta.items()]
    out = bytearray(b'ARROW1\x00\x00')
    out += _message(1, schema, 0)
    dict_blocks, batch_blocks = [], []
    for name, spec, _ in columns:
        if spec[0] == 'dict':
            rb, body = _record_batch([('utf8',)], len(spec[3]), [spec[3]])
            meta = _message(2, {0: ('q', spec[2]), 1: rb, 2: ('?', False)}, len(body))
            dict_blocks.append((len(out), len(meta), 0, len(body)))
            out += meta + body
    specs = [s for _, s, _ in columns]
    for cols in batches:
        rb, body = _record_batch(specs, len(cols[0]), cols, compressed_body)
        meta = _message(3, rb, len(body))
        batch_blocks.append((len(out), len(meta), 0, len(body)))
        out += meta + body
    footer = flatbuffer({0: ('h', 4), 1: schema, 2: Structs('qiiq', dict_blocks), 3: Structs('qiiq', batch_blocks)})
    out += footer + struct.pack('<i', len(footer)) + b'ARROW1'
    return bytes(out)


# ---------------------------------------------------------------------------------------------------
# POD5
# ---------------------------------------------------------------------------------------------------
def container(path: str, tables: Dict[int, bytes], marker: bytes = b'\x5a' * 16) -> None:
    """The POD5 container around embedded Arrow files {content type: bytes}."""
    out = bytearray(SIGNATURE + marker)
    contents = []
    for ctype, data in tables.items():
        contents.append({0: ('q', len(out)), 1: ('q', len(data)), 2: ('h', 0), 3: ('h', ctype)})
        out += data + bytes(-len(data) % 8) + marker
    footer = flatbuffer({0: str(uuid.UUID(bytes=marker)), 1: 'warpstr-b200 tests', 2: '0.3.10', 3: contents})
    out += b'FOOTER\x00\x00' + footer + struct.pack('<q', len(footer)) + marker + SIGNATURE
    with open(path, 'wb') as fh:
        fh.write(out)


UUID = {'ARROW:extension:name': 'minknow.uuid', 'ARROW:extension:metadata': ''}
VBZ = {'ARROW:extension:name': 'minknow.vbz', 'ARROW:extension:metadata': ''}
SCHEMA_META = {'MINKNOW:pod5_version': '0.3.10', 'MINKNOW:software': 'warpstr-b200 tests',
               'MINKNOW:file_identifier': '5a5a5a5a-5a5a-5a5a-5a5a-5a5a5a5a5a5a'}


def _batched(n: int, size: int):
    return [(a, min(a + size, n)) for a in range(0, n, size)] or [(0, 0)]


def write(path: str, reads: Dict[str, np.ndarray], rows: int = 1, seed: int = 0, shuffle: bool = False,
          signal_batch: int = 1 << 30, reads_batch: int = 1 << 30, compressed: bool = True,
          num_samples: bool = True, extra_columns: bool = True, run_info: bool = True,
          compress: Optional[Callable[[bytes], bytes]] = None, tamper: Optional[Callable[[dict], None]] = None,
          compressed_body: bool = False, big_endian: bool = False, more_columns: Sequence[tuple] = ()) -> dict:
    """A POD5 file holding ``reads`` {read ID: int16 samples}.  Every read is cut into ``rows`` signal rows (or
    ``rows(k, n)`` rows for read k of n samples) at random points; ``shuffle`` scatters all rows over the Signal
    table, so a read's rows are neither contiguous nor in order there.  The tables are written in batches of
    ``signal_batch`` / ``reads_batch`` rows.  ``compress``: body -> zstd frame (default ``_h5write.zstd_compress``
    at level 1, as POD5 writes it).  ``tamper`` gets the table contents (see the returned dict) before they are
    written; ``compressed_body`` and ``big_endian`` mark the Signal table so, ``more_columns`` [(name, spec,
    values)] are added to the Reads table.  Returns those contents, and the embedded Arrow files under 'arrow'
    {content type: bytes}."""
    rng = np.random.default_rng(seed)
    compress = compress or hw.zstd_compress
    pieces = []                                             # (read index, samples)
    read_rows = []
    for k, x in enumerate(reads.values()):
        x = np.ascontiguousarray(x, dtype=np.int16)
        m = rows(k, len(x)) if callable(rows) else rows
        cuts = np.sort(rng.integers(0, len(x) + 1, size=m - 1)) if m > 1 else np.zeros(0, np.int64)
        bounds = [0] + cuts.tolist() + [len(x)]
        read_rows.append([])
        for a, b in zip(bounds[:-1], bounds[1:]):
            read_rows[-1].append(len(pieces))
            pieces.append((k, x[a:b]))
    order = rng.permutation(len(pieces)) if shuffle else np.arange(len(pieces))
    where = np.empty(len(pieces), dtype=np.int64)
    where[order] = np.arange(len(pieces))
    ids = [uuid.UUID(r).bytes for r in reads]
    t = dict(read_ids=list(ids),
             read_rows=[[int(where[p]) for p in rr] for rr in read_rows],
             num_samples=[len(np.asarray(x)) for x in reads.values()],
             sig_read_ids=[ids[pieces[p][0]] for p in order],
             sig_samples=[len(pieces[p][1]) for p in order],
             sig_payload=[compress(hw.svb_body(pieces[p][1], 1)) if compressed else pieces[p][1] for p in order])
    if tamper is not None:
        tamper(t)
    sig_spec = ('large_binary',) if compressed else ('large_list', ('int', 16, True))
    sig_cols = [('read_id', ('fsb', 16), UUID), ('signal', sig_spec, VBZ if compressed else None),
                ('samples', ('int', 32, False), None)]
    n_sig = len(t['sig_samples'])
    signal = arrow_file(sig_cols, [[t['sig_read_ids'][a:b], t['sig_payload'][a:b], t['sig_samples'][a:b]]
                                   for a, b in _batched(n_sig, signal_batch)], SCHEMA_META, compressed_body,
                        big_endian)
    n = len(t['read_ids'])
    read_cols = [('read_id', ('fsb', 16), UUID), ('signal', ('list', ('int', 64, False)), None)]
    extra = []
    if extra_columns:
        read_cols += [('read_number', ('int', 32, False), None), ('start', ('int', 64, False), None),
                      ('median_before', ('float', 32), None),
                      ('pore_type', ('dict', 16, 0, ['not_set', 'R9.4.1']), None),
                      ('calibration', ('struct', [('offset', ('float', 32)), ('scale', ('float', 32))]), None),
                      ('end_reason', ('dict', 16, 1, ['unknown', 'signal_positive', 'data_service_unblock_mux_change']),
                       None),
                      ('end_reason_forced', ('bool',), None),
                      ('run_info', ('dict', 16, 2, ['acq0']), None)]
        extra = [np.arange(n) + 100, np.arange(n) * 4000, rng.random(n) * 200, np.arange(n) % 2,
                 {'offset': np.full(n, -240.0), 'scale': np.full(n, 0.1755)}, np.arange(n) % 3, np.arange(n) % 2 == 1,
                 np.zeros(n)]
    for name, spec, values in more_columns:
        read_cols.append((name, spec, None))
        extra.append(values)
    if num_samples:
        read_cols.append(('num_samples', ('int', 64, False), None))
        extra.append(t['num_samples'])

    def cut(col, a, b):
        return {k: v[a:b] for k, v in col.items()} if isinstance(col, dict) else col[a:b]
    reads_tab = arrow_file(read_cols, [[t['read_ids'][a:b], t['read_rows'][a:b]] + [cut(c, a, b) for c in extra]
                                       for a, b in _batched(n, reads_batch)], SCHEMA_META)
    tables = {SIGNAL_TABLE: signal, READS_TABLE: reads_tab}
    if run_info:
        tables[RUN_INFO_TABLE] = arrow_file([('acquisition_id', ('utf8',), None),
                                             ('sample_rate', ('int', 16, False), None),
                                             ('sequencer_position', ('utf8',), None)],
                                            [[['acq0'], [4000], ['MN00000']]], SCHEMA_META)
    container(path, tables)
    t['arrow'] = tables
    return t
