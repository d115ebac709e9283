"""Test helper: writes the small part of HDF5 that warpstr_b200/fast5.py parses, so the reader can be
tested on files without h5py.

* superblock version 0, version-1 object headers;
* groups as a symbol table (v1 group B-tree -> SNOD -> local heap) or as link messages in the header;
* one-dimensional int16 datasets, chunked (v1 chunk B-tree, one or two levels, the last chunk partial and
  coded whole, as HDF5 writes it) through VBZ (the reference's cd_values: version, integer size 2, zig-zag,
  zstd level), deflate + shuffle, or no filter; contiguous datasets.

Layouts: multi-read (``read_<id>/Raw/Signal``) and single-read (``Raw/Reads/Read_<n>/Signal``).
The VBZ encoder follows the published format (nanoporetech/vbz_compression); it is a vectorised restatement
of the one in tests/test_fast5.py.
"""
import ctypes
import struct
import zlib
from typing import Dict, List, Optional, Tuple

import numpy as np

from warpstr_b200 import fast5

VBZ = 32020


def zstd_compress(data: bytes, level: int = 1) -> bytes:
    lib = fast5._libzstd()
    lib.ZSTD_compressBound.restype = ctypes.c_size_t
    lib.ZSTD_compressBound.argtypes = [ctypes.c_size_t]
    lib.ZSTD_compress.restype = ctypes.c_size_t
    lib.ZSTD_compress.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int]
    cap = lib.ZSTD_compressBound(len(data))
    out = ctypes.create_string_buffer(cap)
    n = lib.ZSTD_compress(out, cap, data, len(data), level)
    assert not lib.ZSTD_isError(n)
    return out.raw[:n]


def svb_body(x: np.ndarray, version: int, zigzag: bool = True) -> bytes:
    """int16 samples -> the StreamVByte body of one VBZ chunk (before zstd)."""
    x = np.asarray(x, dtype=np.int64)
    n = len(x)
    if zigzag:
        d = np.diff(x, prepend=0)
        if version == 0:
            d = ((d + 2 ** 31) % 2 ** 32) - 2 ** 31
            v = ((d << 1) ^ (d >> 31)) & 0xFFFFFFFF
        else:
            d = ((d + 32768) % 65536) - 32768      # 16-bit arithmetic wraps
            v = ((d << 1) ^ (d >> 15)) & 0xFFFF
    else:
        v = x & 0xFFFF
    if version == 0:
        nb = 1 + (v >= 1 << 8) + (v >= 1 << 16) + (v >= 1 << 24)
        codes = np.zeros((n + 3) // 4 * 4, dtype=np.uint8)
        codes[:n] = nb - 1
        ctrl = (codes.reshape(-1, 4) << np.array([0, 2, 4, 6], dtype=np.uint8)).sum(axis=1).astype(np.uint8)
        b = v.astype('<u4').view(np.uint8).reshape(n, 4)
        data = b[np.arange(4)[None, :] < nb[:, None]]
    else:
        nb = 1 + (v >= 1 << 8)
        ctrl = np.packbits((nb - 1).astype(np.uint8), bitorder='little')
        b = v.astype('<u2').view(np.uint8).reshape(n, 2)
        data = b[np.arange(2)[None, :] < nb[:, None]]
    return ctrl.tobytes() + data.tobytes()


def vbz_chunk(x: np.ndarray, version: int, zstd: bool = True, zigzag: bool = True) -> bytes:
    """int16 samples -> one chunk as the VBZ filter stores it: uint32 byte size, then the (zstd) body."""
    body = svb_body(x, version, zigzag)
    return struct.pack('<I', 2 * len(x)) + (zstd_compress(body) if zstd else body)


def _pad8(b: bytes) -> bytes:
    return b + bytes(-len(b) % 8)


class _File:
    def __init__(self):
        self.buf = bytearray(96)                   # superblock + root symbol-table entry

    def put(self, data: bytes, align: int = 8) -> int:
        self.buf += bytes(-len(self.buf) % align)
        at = len(self.buf)
        self.buf += data
        return at

    def header(self, messages: List[Tuple[int, bytes]]) -> int:
        """Version-1 object header holding ``messages`` [(type, body)]."""
        body = b''.join(struct.pack('<HHB3x', t, len(_pad8(m)), 0) + _pad8(m) for t, m in messages)
        return self.put(struct.pack('<BBHII', 1, 0, len(messages), 1, len(body)) + bytes(4) + body)

    # -- groups -----------------------------------------------------------------------------------
    def link_group(self, members: Dict[str, int]) -> int:
        msgs = []
        for name, addr in members.items():
            nm = name.encode()
            msgs.append((0x0006, bytes([1, 0, len(nm)]) + nm + struct.pack('<Q', addr)))
        return self.header(msgs)

    def symtab_group(self, members: Dict[str, int]) -> int:
        names = sorted(members)
        heap_data = bytearray(8)                   # offset 0: the empty name
        offs = []
        for nm in names:
            offs.append(len(heap_data))
            heap_data += _pad8(nm.encode() + b'\x00')
        data_addr = self.put(bytes(heap_data))
        heap = self.put(b'HEAP' + bytes([0, 0, 0, 0]) + struct.pack('<QQQ', len(heap_data), UNDEF_ADDR, data_addr))
        snod = b'SNOD' + bytes([1, 0]) + struct.pack('<H', len(names))
        for o, nm in zip(offs, names):
            snod += struct.pack('<QQII', o, members[nm], 0, 0) + bytes(16)
        snod_addr = self.put(snod)
        tree = b'TREE' + bytes([0, 0]) + struct.pack('<HQQ', 1, UNDEF_ADDR, UNDEF_ADDR)
        tree += struct.pack('<QQQ', 0, snod_addr, offs[-1] if offs else 0)
        bt = self.put(tree)
        return self.header([(0x0011, struct.pack('<QQ', bt, heap))])

    # -- datasets ---------------------------------------------------------------------------------
    def dataset(self, x: np.ndarray, filt: str = 'vbz0', chunk: int = 4096, fanout: int = 0) -> int:
        """``filt``: 'vbz0' / 'vbz1' (zstd), 'vbz0-raw' / 'vbz1-raw' (no zstd), 'vbz0-nozz' (no zig-zag),
        'deflate' (shuffle + deflate), 'none' (chunked, no filter), 'contiguous'.  ``fanout`` > 0 spreads the
        chunks over leaf nodes of that many entries under one root node."""
        x = np.ascontiguousarray(x, dtype='<i2')
        n = len(x)
        msgs = [(0x0001, struct.pack('<BBBB4xQ', 1, 1, 0, 0, n)),
                (0x0003, struct.pack('<BBBBIHH', 0x10, 0x08, 0, 0, 2, 0, 16))]
        if filt == 'contiguous':
            addr = self.put(x.tobytes())
            msgs.append((0x0008, struct.pack('<BBQQ', 3, 1, addr, 2 * n)))
            return self.header(msgs)
        entries = []
        for start in range(0, n, chunk):
            part = np.zeros(chunk, dtype='<i2')
            part[:min(chunk, n - start)] = x[start:start + chunk]      # a partial last chunk is stored whole
            if filt.startswith('vbz'):
                data = vbz_chunk(part, int(filt[3]), zstd=not filt.endswith('-raw'), zigzag=not filt.endswith('-nozz'))
            elif filt == 'deflate':
                data = zlib.compress(part.view(np.uint8).reshape(-1, 2).T.tobytes())
            else:
                data = part.tobytes()
            entries.append((start, len(data), self.put(data)))
        if filt.startswith('vbz'):
            version = int(filt[3])
            zz = 0 if filt.endswith('-nozz') else 1
            pipeline = [(VBZ, b'vbz', (version, 2, zz, 0 if filt.endswith('-raw') else 1))]
        elif filt == 'deflate':
            pipeline = [(2, b'shuffle', (2,)), (1, b'deflate', (4,))]
        else:
            pipeline = []
        bt = self._chunk_btree(entries, chunk, fanout)
        msgs.append((0x0008, struct.pack('<BBBQII', 3, 2, 2, bt, chunk, 2)))
        if pipeline:
            fp = bytes([1, len(pipeline)]) + bytes(6)
            for fid, name, cd in pipeline:
                nm = _pad8(name + b'\x00')
                fp += struct.pack('<HHHH', fid, len(nm), 0, len(cd)) + nm + struct.pack('<%dI' % len(cd), *cd)
                if len(cd) % 2:
                    fp += bytes(4)
            msgs.append((0x000B, fp))
        return self.header(msgs)

    def _chunk_btree(self, entries, chunk: int, fanout: int) -> int:
        def node(level, items):           # items: [(first element, stored bytes, child address)]
            out = b'TREE' + bytes([1, level]) + struct.pack('<HQQ', len(items), UNDEF_ADDR, UNDEF_ADDR)
            for start, size, child in items:
                out += struct.pack('<IIQQ', size, 0, start, 0) + struct.pack('<Q', child)
            last = items[-1][0] + chunk if items else 0
            out += struct.pack('<IIQQ', 0, 0, last, 0)
            return self.put(out)
        if fanout <= 0 or len(entries) <= fanout:
            return node(0, entries)
        leaves = [(entries[i][0], 0, node(0, entries[i:i + fanout])) for i in range(0, len(entries), fanout)]
        return node(1, leaves)

    def finish(self, root: int) -> bytes:
        b = self.buf
        b[0:8] = b'\x89HDF\r\n\x1a\n'
        b[8:16] = bytes([0, 0, 0, 0, 0, 8, 8, 0])
        b[16:24] = struct.pack('<HHI', 4, 16, 0)
        b[24:56] = struct.pack('<QQQQ', 0, UNDEF_ADDR, len(b), UNDEF_ADDR)
        b[56:96] = struct.pack('<QQII', 0, root, 0, 0) + bytes(16)
        return bytes(b)


UNDEF_ADDR = 0xFFFFFFFFFFFFFFFF


def write_multi(path: str, reads: Dict[str, np.ndarray], filt: str = 'vbz0', chunk: int = 4096,
                root: str = 'symtab', fanout: int = 0) -> None:
    """A multi-read fast5: ``read_<id>/Raw/Signal`` for every (id, samples) of ``reads``."""
    f = _File()
    members = {}
    for rid, x in reads.items():
        sig = f.dataset(x, filt, chunk, fanout)
        members['read_' + rid] = f.link_group({'Raw': f.link_group({'Signal': sig})})
    top = f.symtab_group(members) if root == 'symtab' else f.link_group(members)
    with open(path, 'wb') as fh:
        fh.write(f.finish(top))


def write_single(path: str, x: np.ndarray, read_number: int = 7, filt: str = 'vbz0', chunk: int = 4096,
                 root: str = 'links') -> None:
    """A single-read fast5: ``Raw/Reads/Read_<n>/Signal``."""
    f = _File()
    sig = f.dataset(x, filt, chunk)
    reads = f.link_group({f'Read_{read_number}': f.link_group({'Signal': sig})})
    raw = f.link_group({'Reads': reads})
    top = f.symtab_group({'Raw': raw}) if root == 'symtab' else f.link_group({'Raw': raw})
    with open(path, 'wb') as fh:
        fh.write(f.finish(top))


def corrupt_vbz_chunk(path: str, read_id: str, which: int = 0) -> None:
    """Rewrite the codes of chunk ``which`` of a read written with 'vbz0-raw' or 'vbz1-raw' (no zstd) in place
    so that every value claims the widest form: the data block is then too short for the codes, the error a
    truncated or damaged file gives."""
    with fast5.H5File(path) as h5:
        obj = h5._object(h5._resolve(f'read_{read_id}/Raw/Signal'))
        version = obj.filters[0][1][0]
        _, _, _, addr = sorted(h5._chunk_entries(obj))[which]
        (size,) = struct.unpack_from('<I', h5.buf, addr)
    n = size // 2
    n_ctrl = (n + 3) // 4 if version == 0 else (n + 7) // 8
    with open(path, 'r+b') as fh:
        fh.seek(addr + 4)
        fh.write(b'\xff' * n_ctrl)
