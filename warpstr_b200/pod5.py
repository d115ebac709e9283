"""Minimal POD5 reader: just enough of the container and of Arrow IPC to pull a read's signal rows.

POD5 is the raw-signal format ONT's current software writes.  Like ``fast5.py``, which reads HDF5 without h5py,
this module reads POD5 without the ``pod5`` or ``pyarrow`` packages, and only what the caller needs:

* The container (POD5 0.x): an 8-byte signature, a 16-byte section marker, the embedded Arrow IPC files (each
  followed by zero padding to 8 bytes and the marker), ``FOOTER\\0\\0``, a flatbuffer footer (``footer.fbs``,
  ``Minknow.ReadsFormat``) listing where each embedded file is, the footer's length, the marker and the signature.
* Arrow IPC files as far as the two tables need: the file footer's schema and record-batch blocks, encapsulated
  ``RecordBatch`` messages, their field nodes and buffers.  Columns that are not used are skipped by the node and
  buffer counts of their types; dictionary batches are not decoded.  Big-endian schemas, compressed bodies
  (``BodyCompression``) and types outside the table in ``_layout`` are refused.
* The Signal table (``read_id``, ``signal``, ``samples``) and the Reads table (``read_id``, ``signal``: the read's
  global rows in the Signal table, and ``num_samples`` where the file has it).

A compressed signal row is what VBZ version 1 makes of 2-byte integers (zig-zag deltas, StreamVByte-16 keys and
data) in one zstd frame, without fast5's 4-byte size header; the sample count is the row's ``samples``.  So a row is
one ``RawChunk`` of kind ``KIND_VBZ1_ZSTD`` and takes the same device chain as a fast5 VBZ chunk.  An uncompressed
row (``large_list<int16>``) is a ``KIND_RAW`` chunk.

A read ID is the canonical lower-case hyphenated UUID of the 16 stored bytes, the name fast5 files give a read
after ``read_``.  ``fast5.open_raw`` picks this reader or the HDF5 one from a file's first 8 bytes.
"""
import mmap
import struct
from typing import Dict, List, Optional, Tuple

import numpy as np

from .fast5 import (KIND_RAW, KIND_VBZ1, KIND_VBZ1_ZSTD, CompressedRead, Fast5FormatError, RawChunk,
                    zstd_decompress, zstd_frame_size)

SIGNATURE = b'\x8bPOD\r\n\x1a\n'
FOOTER_MAGIC = b'FOOTER\x00\x00'
ARROW_MAGIC = b'ARROW1'
READS_TABLE, SIGNAL_TABLE = 0, 1                # EmbeddedFile.content_type (2-4: indices, run info: unused)


class Pod5FormatError(Fast5FormatError):
    pass


# ---------------------------------------------------------------------------------------------------
# flatbuffers (little-endian): a table starts with the signed offset back to its vtable
# ---------------------------------------------------------------------------------------------------
class _Table:
    __slots__ = ('b', 't', 'vt', 'vlen')

    def __init__(self, b: bytes, t: int):
        self.b, self.t = b, t
        self.vt = t - struct.unpack_from('<i', b, t)[0]
        self.vlen = struct.unpack_from('<H', b, self.vt)[0]

    @classmethod
    def root(cls, b: bytes) -> '_Table':
        return cls(b, struct.unpack_from('<I', b, 0)[0])

    def _field(self, i: int) -> int:
        o = 4 + 2 * i
        return struct.unpack_from('<H', self.b, self.vt + o)[0] if o + 2 <= self.vlen else 0

    def scalar(self, i: int, fmt: str, default=0):
        o = self._field(i)
        return struct.unpack_from('<' + fmt, self.b, self.t + o)[0] if o else default

    def _target(self, i: int) -> Optional[int]:
        o = self._field(i)
        if not o:
            return None
        p = self.t + o
        return p + struct.unpack_from('<I', self.b, p)[0]

    def table(self, i: int) -> Optional['_Table']:
        p = self._target(i)
        return None if p is None else _Table(self.b, p)

    def string(self, i: int) -> Optional[str]:
        p = self._target(i)
        if p is None:
            return None
        (n,) = struct.unpack_from('<I', self.b, p)
        if p + 4 + n > len(self.b):
            raise struct.error('string past the buffer')
        return bytes(self.b[p + 4:p + 4 + n]).decode('utf-8')

    def tables(self, i: int) -> List['_Table']:
        p = self._target(i)
        if p is None:
            return []
        (n,) = struct.unpack_from('<I', self.b, p)
        return [_Table(self.b, q + struct.unpack_from('<I', self.b, q)[0]) for q in range(p + 4, p + 4 + 4 * n, 4)]

    def structs(self, i: int, fmt: str) -> List[tuple]:
        p = self._target(i)
        if p is None:
            return []
        (n,) = struct.unpack_from('<I', self.b, p)
        size = struct.calcsize('<' + fmt)
        if p + 4 + n * size > len(self.b):
            raise struct.error('vector past the buffer')
        return list(struct.iter_unpack('<' + fmt, self.b[p + 4:p + 4 + n * size])) if n else []


# ---------------------------------------------------------------------------------------------------
# Arrow IPC file format (Schema.fbs, Message.fbs, File.fbs)
# ---------------------------------------------------------------------------------------------------
T_NULL, T_INT, T_FLOAT, T_BINARY, T_UTF8, T_BOOL = 1, 2, 3, 4, 5, 6
T_LIST, T_STRUCT, T_FIXED_SIZE_BINARY, T_FIXED_SIZE_LIST = 12, 13, 15, 16
T_LARGE_BINARY, T_LARGE_UTF8, T_LARGE_LIST = 19, 20, 21
_FIXED_WIDTH = {T_INT, T_FLOAT, T_BOOL, 7, 8, 9, 10, 11, T_FIXED_SIZE_BINARY, 18}   # + Decimal, Date, Time,
_VAR_WIDTH = {T_BINARY, T_UTF8, T_LARGE_BINARY, T_LARGE_UTF8}                       # Timestamp, Interval, Duration
_MSG_RECORD_BATCH = 3


class _Field:
    """A schema field: its name, type id and type table, children, whether it is dictionary-encoded."""

    def __init__(self, fb: _Table):
        self.name = fb.string(0) or ''
        self.type_id = fb.scalar(2, 'B')
        self.type = fb.table(3)
        self.dictionary = fb.table(4) is not None
        self.children = [_Field(c) for c in fb.tables(5)]

    def int_type(self) -> Tuple[int, bool]:
        return (self.type.scalar(0, 'i'), bool(self.type.scalar(1, '?'))) if self.type is not None else (0, False)


def _layout(f: _Field, where: str) -> Tuple[int, int]:
    """(field nodes, buffers) a column of this field takes in a record batch, its children included."""
    if f.dictionary:                                    # laid out as its index type, an Int
        return 1, 2
    t = f.type_id
    if t in _FIXED_WIDTH:
        return 1, 2
    if t in _VAR_WIDTH:
        return 1, 3
    if t == T_NULL:
        return 1, 0
    if t in (T_LIST, T_LARGE_LIST, T_FIXED_SIZE_LIST, T_STRUCT):
        if t != T_STRUCT and len(f.children) != 1:
            raise Pod5FormatError(f'{where}: list column {f.name!r} needs exactly one child')
        nodes, bufs = 1, 1 if t in (T_FIXED_SIZE_LIST, T_STRUCT) else 2
        for c in f.children:
            cn, cb = _layout(c, where)
            nodes, bufs = nodes + cn, bufs + cb
        return nodes, bufs
    raise Pod5FormatError(f'{where}: column {f.name!r} has Arrow type {t}, which this reader does not support')


class _Column:
    """One column of one record batch: absolute (offset, length) of its buffers in the file, its length and nulls."""
    __slots__ = ('field', 'length', 'nulls', 'buffers', 'child_nulls')

    def __init__(self, field, length, nulls, buffers, child_nulls):
        self.field, self.length, self.nulls, self.buffers, self.child_nulls = field, length, nulls, buffers, child_nulls


class _ArrowFile:
    """The schema and record batches of one embedded Arrow IPC file; columns by name, per batch."""

    def __init__(self, buf, start: int, length: int, where: str):
        self.where = where
        end = start + length
        if length < 18 or buf[start:start + 8] != ARROW_MAGIC + b'\x00\x00' or buf[end - 6:end] != ARROW_MAGIC:
            raise Pod5FormatError(f'{where}: not an Arrow IPC file (magic missing at its start or end)')
        (flen,) = struct.unpack_from('<i', buf, end - 10)
        if flen <= 0 or end - 10 - flen < start + 8:
            raise Pod5FormatError(f'{where}: bad Arrow footer length {flen}')
        footer = _Table.root(buf[end - 10 - flen:end - 10])
        schema = footer.table(1)
        if schema is None:
            raise Pod5FormatError(f'{where}: Arrow footer without a schema')
        if schema.scalar(0, 'h') != 0:
            raise Pod5FormatError(f'{where}: big-endian Arrow schemas are not supported')
        self.fields = [_Field(f) for f in schema.tables(1)]
        self.layouts = [_layout(f, where) for f in self.fields]
        self.batches: List[Tuple[int, Dict[str, _Column]]] = []
        for off, meta_len, body_len in footer.structs(3, 'qi4xq'):
            self.batches.append(self._batch(buf, start, end, start + off, meta_len, body_len))

    def _batch(self, buf, start, end, at, meta_len, body_len):
        where = self.where
        if at < start or at + meta_len + body_len > end or meta_len < 8:
            raise Pod5FormatError(f'{where}: record batch block outside the file')
        cont, n = struct.unpack_from('<Ii', buf, at)
        p = at + 8
        if cont != 0xFFFFFFFF or n <= 0 or p + n > at + meta_len:
            raise Pod5FormatError(f'{where}: bad encapsulated message header')
        msg = _Table.root(buf[p:p + n])
        if msg.scalar(1, 'B') != _MSG_RECORD_BATCH:
            raise Pod5FormatError(f'{where}: a record batch block does not hold a RecordBatch message')
        rb = msg.table(2)
        if rb.table(3) is not None:
            raise Pod5FormatError(f'{where}: compressed Arrow record batch bodies (BodyCompression) are not supported')
        length = rb.scalar(0, 'q')
        nodes = rb.structs(1, 'qq')
        bufs = rb.structs(2, 'qq')
        if len(nodes) != sum(l[0] for l in self.layouts) or len(bufs) != sum(l[1] for l in self.layouts):
            raise Pod5FormatError(f'{where}: record batch node/buffer counts do not match the schema')
        body = at + meta_len
        for o, ln in bufs:
            if o < 0 or ln < 0 or o + ln > body_len:
                raise Pod5FormatError(f'{where}: record batch buffer outside its body')
        cols, ni, bi = {}, 0, 0
        for f, (nn, nb) in zip(self.fields, self.layouts):
            cols[f.name] = _Column(f, nodes[ni][0], nodes[ni][1], [(body + o, ln) for o, ln in bufs[bi:bi + nb]],
                                   [nd[1] for nd in nodes[ni + 1:ni + nn]])
            ni, bi = ni + nn, bi + nb
        return length, cols


# ---------------------------------------------------------------------------------------------------
# POD5
# ---------------------------------------------------------------------------------------------------
def _uuid(b: bytes) -> str:
    h = b.hex()
    return f'{h[:8]}-{h[8:12]}-{h[12:16]}-{h[16:20]}-{h[20:32]}'


def _uuids(ids: np.ndarray) -> List[str]:
    """(n, 16) uint8 -> canonical UUID strings."""
    h = ids.tobytes().hex()
    return [f'{h[k:k + 8]}-{h[k + 8:k + 12]}-{h[k + 12:k + 16]}-{h[k + 16:k + 20]}-{h[k + 20:k + 32]}'
            for k in range(0, len(h), 32)]


class Pod5File:
    """An open POD5 file: mmapped, its footer and both tables parsed and every read's rows indexed once."""

    def __init__(self, path: str):
        self.path = path
        self._fh = open(path, 'rb')
        try:
            self.buf = mmap.mmap(self._fh.fileno(), 0, access=mmap.ACCESS_READ)
        except ValueError as exc:
            self._fh.close()
            raise Pod5FormatError(f'{path}: empty file') from exc
        try:
            self._parse()
        except (struct.error, IndexError, UnicodeDecodeError) as exc:
            self.close()
            raise Pod5FormatError(f'{path}: malformed POD5 metadata ({exc})') from exc
        except Exception:
            self.close()
            raise

    def close(self):
        try:
            self.buf.close()
        finally:
            self._fh.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _bytes(self, a: int, n: int) -> bytes:
        if a < 0 or a + n > len(self.buf):
            raise Pod5FormatError(f'{self.path}: Arrow buffer outside the file')
        return self.buf[a:a + n]

    # -- container ---------------------------------------------------------------------------------
    def _parse(self):
        b, path = self.buf, self.path
        size = len(b)
        if size < 8 or b[:8] != SIGNATURE:
            raise Pod5FormatError(f'{path}: not a POD5 file (bad signature)')
        if size < 24 + 8 + 8 + 16 + 8:
            raise Pod5FormatError(f'{path}: truncated POD5 file')
        marker = b[8:24]
        if b[size - 8:] != SIGNATURE or b[size - 24:size - 8] != marker:
            raise Pod5FormatError(f'{path}: truncated POD5 file (no closing signature and section marker)')
        pos = size - 32
        (flen,) = struct.unpack_from('<q', b, pos)
        start = pos - (flen + 7) // 8 * 8                  # the flatbuffer is padded to 8 bytes before its length
        if flen <= 0 or start < 32 or b[start - 8:start] != FOOTER_MAGIC:
            raise Pod5FormatError(f'{path}: truncated or bad POD5 footer (footer length {flen})')
        footer = _Table.root(b[start:pos])
        tables = {}
        for ef in footer.tables(3):
            off, ln, fmt, ctype = ef.scalar(0, 'q'), ef.scalar(1, 'q'), ef.scalar(2, 'h'), ef.scalar(3, 'h')
            if ctype not in (READS_TABLE, SIGNAL_TABLE):
                continue
            if fmt != 0:
                raise Pod5FormatError(f'{path}: embedded file format {fmt} is not Feather V2 / Arrow IPC')
            if ctype in tables:
                raise Pod5FormatError(f'{path}: more than one {"reads" if ctype == READS_TABLE else "signal"} table')
            if off < 24 or ln <= 0 or off + ln > start - 8:
                raise Pod5FormatError(f'{path}: embedded file outside the file')
            tables[ctype] = _ArrowFile(b, off, ln, f'{path}: {"reads" if ctype == READS_TABLE else "signal"} table')
        for ctype, name in ((SIGNAL_TABLE, 'signal'), (READS_TABLE, 'reads')):
            if ctype not in tables:
                raise Pod5FormatError(f'{path}: no {name} table in the footer')
        self._signal_table(tables[SIGNAL_TABLE])
        self._reads_table(tables[READS_TABLE])
        self._index()

    # -- column readers ----------------------------------------------------------------------------
    def _col(self, t: _ArrowFile, cols: Dict[str, _Column], name: str, required: bool = True) -> Optional[_Column]:
        c = cols.get(name)
        if c is None:
            if required:
                raise Pod5FormatError(f'{t.where}: no {name!r} column')
            return None
        if c.nulls or any(c.child_nulls):
            raise Pod5FormatError(f'{t.where}: column {name!r} has null values')
        return c

    def _uuid_col(self, t, c: _Column) -> np.ndarray:
        f = c.field
        if f.dictionary or f.type_id != T_FIXED_SIZE_BINARY or f.type.scalar(0, 'i') != 16:
            raise Pod5FormatError(f'{t.where}: column {f.name!r} is not a 16-byte UUID column')
        a, ln = c.buffers[1]
        if ln < 16 * c.length:
            raise Pod5FormatError(f'{t.where}: column {f.name!r} is shorter than its rows')
        return np.frombuffer(self._bytes(a, 16 * c.length), dtype=np.uint8).reshape(c.length, 16)

    def _values(self, t, c: _Column, buf: int, count: int, dtype: str) -> np.ndarray:
        a, ln = c.buffers[buf]
        n = count * np.dtype(dtype).itemsize
        if ln < n:
            raise Pod5FormatError(f'{t.where}: column {c.field.name!r} is shorter than its rows')
        return np.frombuffer(self._bytes(a, n), dtype=dtype)

    def _uint_col(self, t, c: _Column, bits: Tuple[int, ...]) -> np.ndarray:
        f = c.field
        w, signed = f.int_type()
        if f.dictionary or f.type_id != T_INT or signed or w not in bits:
            raise Pod5FormatError(f'{t.where}: column {f.name!r} is not an unsigned integer column')
        return self._values(t, c, 1, c.length, f'<u{w // 8}').astype(np.int64)

    def _signal_table(self, t: _ArrowFile):
        ids, samples, lo, hi, compressed = [], [], [], [], None
        for length, cols in t.batches:
            rid = self._uuid_col(t, self._col(t, cols, 'read_id'))
            ns = self._uint_col(t, self._col(t, cols, 'samples'), (32, 64))
            sig = self._col(t, cols, 'signal')
            f = sig.field
            if f.type_id == T_LARGE_BINARY and not f.dictionary:
                offs = self._values(t, sig, 1, length + 1, '<i8')
                data_at, data_len = sig.buffers[2]
                kind = True
            elif (f.type_id == T_LARGE_LIST and not f.dictionary and f.children[0].type_id == T_INT
                  and f.children[0].int_type() == (16, True) and not f.children[0].dictionary):
                offs = self._values(t, sig, 1, length + 1, '<i8') * 2
                data_at, data_len = sig.buffers[3]
                kind = False
            else:
                raise Pod5FormatError(f'{t.where}: signal column is neither large_binary (VBZ) nor '
                                      f'large_list<int16>')
            if compressed is not None and kind != compressed:
                raise Pod5FormatError(f'{t.where}: signal column type changes between batches')
            compressed = kind
            if length and ((np.diff(offs) < 0).any() or offs[0] < 0 or offs[-1] > data_len):
                raise Pod5FormatError(f'{t.where}: signal offsets outside their data buffer')
            ids.append(rid)
            samples.append(ns)
            lo.append(data_at + offs[:-1])
            hi.append(data_at + offs[1:])
        self.compressed = bool(compressed)
        self._sig_id = np.concatenate(ids) if ids else np.zeros((0, 16), np.uint8)
        self._sig_samples, self._sig_lo, self._sig_hi = (np.concatenate(a) if a else np.zeros(0, np.int64)
                                                         for a in (samples, lo, hi))
        if not self.compressed and (self._sig_hi - self._sig_lo != 2 * self._sig_samples).any():
            k = int(np.flatnonzero(self._sig_hi - self._sig_lo != 2 * self._sig_samples)[0])
            raise Pod5FormatError(f'{self.path}: signal row {k} holds {(self._sig_hi[k] - self._sig_lo[k]) // 2} '
                                  f'samples, not its {self._sig_samples[k]}')

    def _reads_table(self, t: _ArrowFile):
        ids, rows, counts, nsamp = [], [], [], []
        has_num = None
        for length, cols in t.batches:
            ids.append(self._uuid_col(t, self._col(t, cols, 'read_id')))
            sig = self._col(t, cols, 'signal')
            f = sig.field
            if f.dictionary or f.type_id not in (T_LIST, T_LARGE_LIST) or f.children[0].type_id != T_INT \
                    or f.children[0].dictionary or f.children[0].int_type()[1] \
                    or f.children[0].int_type()[0] not in (32, 64):
                raise Pod5FormatError(f'{t.where}: signal column is not a list of unsigned row indices')
            offs = self._values(t, sig, 1, length + 1, '<i4' if f.type_id == T_LIST else '<i8').astype(np.int64)
            if length and ((np.diff(offs) < 0).any() or offs[0] < 0):
                raise Pod5FormatError(f'{t.where}: bad signal list offsets')
            n_child = int(offs[-1]) if length else 0
            child = self._values(t, sig, 3, n_child, f'<u{f.children[0].int_type()[0] // 8}')
            rows.append(child[offs[0]:n_child].astype(np.uint64) if length else child[:0].astype(np.uint64))
            counts.append(np.diff(offs))
            num = self._col(t, cols, 'num_samples', required=False)
            if has_num is not None and (num is not None) != has_num:
                raise Pod5FormatError(f'{t.where}: num_samples present in some batches only')
            has_num = num is not None
            if has_num:
                nsamp.append(self._uint_col(t, num, (64, 32)))
        self._read_id = np.concatenate(ids) if ids else np.zeros((0, 16), np.uint8)
        self._rows = np.concatenate(rows) if rows else np.zeros(0, np.uint64)
        self._row_off = np.zeros(len(self._read_id) + 1, dtype=np.int64)
        if counts:
            np.cumsum(np.concatenate(counts), out=self._row_off[1:])
        self._num_samples = np.concatenate(nsamp) if has_num else None

    # -- the read index, with every cross-table check ----------------------------------------------
    def _index(self):
        path = self.path
        names = _uuids(self._read_id)
        self.names = names
        self._by_name = {}
        for k, nm in enumerate(names):
            if nm in self._by_name:
                raise Pod5FormatError(f'{path}: read {nm} appears twice in the reads table')
            self._by_name[nm] = k
        n_sig = len(self._sig_samples)
        owner = np.repeat(np.arange(len(names)), np.diff(self._row_off))
        out = np.flatnonzero(self._rows >= n_sig)
        if len(out):
            k = int(out[0])
            raise Pod5FormatError(f'{path}: read {names[owner[k]]}: signal row {int(self._rows[k])} is out of range '
                                  f'(the signal table has {n_sig} rows)')
        rows = self._rows.astype(np.int64)
        used = np.bincount(rows, minlength=n_sig)
        twice = np.flatnonzero(used > 1)
        if len(twice):
            r = int(twice[0])
            who = sorted({names[owner[k]] for k in np.flatnonzero(rows == r)})
            raise Pod5FormatError(f'{path}: signal row {r} is used more than once, by read(s) {", ".join(who)}')
        wrong = np.flatnonzero((self._sig_id[rows] != self._read_id[owner]).any(axis=1))
        if len(wrong):
            k = int(wrong[0])
            raise Pod5FormatError(f'{path}: read {names[owner[k]]}: signal row {rows[k]} belongs to read '
                                  f'{_uuid(self._sig_id[rows[k]].tobytes())}')
        cs = np.zeros(len(rows) + 1, dtype=np.int64)
        np.cumsum(self._sig_samples[rows], out=cs[1:])
        self._row_start = cs[:-1] - cs[self._row_off[owner]]
        self._n_samples = cs[self._row_off[1:]] - cs[self._row_off[:-1]]
        if self._num_samples is not None:
            bad = np.flatnonzero(self._n_samples != self._num_samples)
            if len(bad):
                k = int(bad[0])
                raise Pod5FormatError(f'{path}: read {names[k]}: its signal rows hold {int(self._n_samples[k])} '
                                      f'samples, num_samples says {int(self._num_samples[k])}')

    # -- reads -------------------------------------------------------------------------------------
    def read_names(self) -> List[str]:
        return list(self.names)

    def _read(self, read_id: Optional[str]) -> int:
        if read_id is None:
            if len(self.names) == 1:
                return 0
            raise Pod5FormatError(f'{self.path}: holds {len(self.names)} reads, so a read ID is needed')
        k = self._by_name.get(str(read_id).strip().lower())
        if k is None:
            raise Pod5FormatError(f'{self.path}: read {read_id} not found')
        return k

    def read_chunks(self, read_id: Optional[str], keep_frames: bool) -> CompressedRead:
        """A read's signal rows as chunks, in the read's row order, starting at the running sum of ``samples``:
        ``keep_frames`` leaves a zstd frame the device decoder takes as it is stored (KIND_VBZ1_ZSTD); any other
        frame is undone here (KIND_VBZ1).  Uncompressed rows are KIND_RAW."""
        k = self._read(read_id)
        chunks = []
        for j in range(int(self._row_off[k]), int(self._row_off[k + 1])):
            r = int(self._rows[j])
            n = int(self._sig_samples[r])
            if n == 0:                          # an empty row adds no samples (and no chunk for the device)
                continue
            payload = self.buf[int(self._sig_lo[r]):int(self._sig_hi[r])]
            start = int(self._row_start[j])
            if not self.compressed:
                chunks.append(RawChunk(start, n, KIND_RAW, payload))
                continue
            size = zstd_frame_size(payload, 5 * n + 16) if keep_frames else -1
            if size >= 0:
                chunks.append(RawChunk(start, n, KIND_VBZ1_ZSTD, payload, True, n, size))
            else:
                chunks.append(RawChunk(start, n, KIND_VBZ1, zstd_decompress(payload, 5 * n + 16), True, n))
        return CompressedRead(self.path, self.names[k], int(self._n_samples[k]), chunks)

    def read_signal(self, read_id: Optional[str]) -> np.ndarray:
        return self.read_chunks(read_id, keep_frames=False).decode()


def read_names(path: str) -> List[str]:
    """Read IDs of a POD5 file, in the reads table's order."""
    with Pod5File(path) as f:
        return f.read_names()


def raw_signal(path: str, read_id: Optional[str] = None) -> np.ndarray:
    """The raw int16 DAC samples of one read (the only read of the file when ``read_id`` is None)."""
    with Pod5File(path) as f:
        return f.read_signal(read_id)


def raw_chunks(path: str, read_id: Optional[str] = None, f: Optional[Pod5File] = None) -> CompressedRead:
    """One read's signal rows with zstd undone on the host (KIND_VBZ1, or KIND_RAW for uncompressed signal); the
    StreamVByte decode is left to the GPU.  ``f``: the file, already open."""
    if f is None:
        with Pod5File(path) as g:
            return g.read_chunks(read_id, keep_frames=False)
    return f.read_chunks(read_id, keep_frames=False)


def stored_chunks(path: str, read_id: Optional[str] = None, f: Optional[Pod5File] = None) -> CompressedRead:
    """``raw_chunks`` with every zstd frame the device decodes (``fast5.zstd_frame_size``) left as stored."""
    if f is None:
        with Pod5File(path) as g:
            return g.read_chunks(read_id, keep_frames=True)
    return f.read_chunks(read_id, keep_frames=True)
