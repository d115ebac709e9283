"""Minimal fast5 reader: just enough HDF5 and VBZ to pull a read's raw int16 signal.

The reference opens fast5 files with h5py and the VBZ HDF5 plugin (schemas/fast5.py:17-18,
50-52; prepare_caller_only.py:78-85).  Neither ships with this build, and the caller needs
exactly one thing from the container -- ``Raw/.../Signal`` -- so this module reads that and
nothing else:

* HDF5 as MinKNOW/ont_fast5_api write it: superblock version 0, version-1 object headers,
  "old style" groups (symbol-table message -> v1 B-tree of SNOD nodes -> local heap) and
  compact "new style" groups (link messages in the header), datasets with contiguous, compact
  or chunked (v1 chunk B-tree) layout.
* Filters: VBZ (id 32020: [uint32 size][zstd frame] -> StreamVByte -> zig-zag delta, versions
  0 and 1 of the 2-byte-integer coding), deflate (1) and shuffle (2) for uncompressed-era files.

Both file flavours are understood: multi-read (``read_<id>/Raw/Signal``, what a sequencing run
or ``test/test_input/*/fast5s`` holds) and single-read (``Raw/Reads/Read_<n>/Signal``, what the
reference's extraction step writes).  libzstd is loaded with ctypes (the image has
libzstd.so.1 but no Python binding).

``Fast5`` mirrors the part of the reference class the caller uses: ``get_data_processed``
sends the raw read through the GPU normalisation kernel (normalize.py).
"""
import ctypes
import ctypes.util
import mmap
import struct
import zlib
from dataclasses import dataclass
from typing import Dict, Iterator, List, NamedTuple, Optional, Tuple

import numpy as np

UNDEF = 0xFFFFFFFFFFFFFFFF
VBZ_FILTER_ID = 32020


class Fast5FormatError(ValueError):
    pass


# ---------------------------------------------------------------------------------------------------
# zstd through ctypes
# ---------------------------------------------------------------------------------------------------
_zstd = None


def _libzstd():
    global _zstd
    if _zstd is None:
        name = ctypes.util.find_library('zstd') or 'libzstd.so.1'
        try:
            lib = ctypes.CDLL(name)
        except OSError as exc:
            raise ImportError('VBZ-compressed fast5 needs libzstd (libzstd.so.1 not loadable)') from exc
        lib.ZSTD_getFrameContentSize.restype = ctypes.c_ulonglong
        lib.ZSTD_getFrameContentSize.argtypes = [ctypes.c_void_p, ctypes.c_size_t]
        lib.ZSTD_decompress.restype = ctypes.c_size_t
        lib.ZSTD_decompress.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t]
        lib.ZSTD_isError.restype = ctypes.c_uint
        lib.ZSTD_isError.argtypes = [ctypes.c_size_t]
        _zstd = lib
    return _zstd


def zstd_decompress(data: bytes, max_size: int) -> bytes:
    lib = _libzstd()
    n = lib.ZSTD_getFrameContentSize(data, len(data))
    if n in (2 ** 64 - 1, 2 ** 64 - 2) or n > max_size:      # unknown / error: fall back to the bound we know
        n = max_size
    out = ctypes.create_string_buffer(max(int(n), 1))
    got = lib.ZSTD_decompress(out, int(n), data, len(data))
    if lib.ZSTD_isError(got):
        raise Fast5FormatError('zstd: corrupt VBZ chunk')
    return out.raw[:got]


# ---------------------------------------------------------------------------------------------------
# VBZ (nanoporetech/vbz_compression): StreamVByte + zig-zag delta
# ---------------------------------------------------------------------------------------------------
def _svb_decode_u32(buf: np.ndarray, n: int) -> np.ndarray:
    """StreamVByte: ceil(n/4) control bytes (2 bits per value, low bits first, code c = c+1 data
    bytes), then the little-endian data bytes."""
    n_ctrl = (n + 3) // 4
    if len(buf) < n_ctrl:
        raise Fast5FormatError('VBZ: truncated StreamVByte control block')
    ctrl = buf[:n_ctrl]
    codes = ((ctrl[:, None] >> np.array([0, 2, 4, 6], dtype=np.uint8)) & 3).reshape(-1)[:n].astype(np.int64)
    lens = codes + 1
    starts = np.zeros(n, dtype=np.int64)
    np.cumsum(lens[:-1], out=starts[1:])
    data = buf[n_ctrl:]
    if n and starts[-1] + lens[-1] > len(data):
        raise Fast5FormatError('VBZ: truncated StreamVByte data block')
    padded = np.concatenate((data, np.zeros(4, dtype=np.uint8))).astype(np.uint32)
    out = padded[starts]
    for k in range(1, 4):
        out = out | np.where(lens > k, padded[starts + k] << np.uint32(8 * k), np.uint32(0))
    return out.astype(np.uint32)


def _svb_decode_u16(buf: np.ndarray, n: int) -> np.ndarray:
    """The 16-bit StreamVByte variant of VBZ version 1: ceil(n/8) key bytes (1 bit per value,
    low bits first: 0 = one data byte, 1 = two), then the data bytes."""
    n_key = (n + 7) // 8
    if len(buf) < n_key:
        raise Fast5FormatError('VBZ: truncated key block')
    bits = np.unpackbits(buf[:n_key], bitorder='little')[:n].astype(np.int64)
    lens = bits + 1
    starts = np.zeros(n, dtype=np.int64)
    np.cumsum(lens[:-1], out=starts[1:])
    data = buf[n_key:]
    if n and starts[-1] + lens[-1] != len(data):
        raise Fast5FormatError('VBZ v1: data block length does not match the keys')
    padded = np.concatenate((data, np.zeros(2, dtype=np.uint8))).astype(np.uint16)
    return (padded[starts] | np.where(lens > 1, padded[starts + 1] << np.uint16(8), np.uint16(0))).astype(np.uint16)


def _vbz_params(cd_values: Tuple[int, ...]):
    """(version, integer size, zig-zag flag, zstd level) of the VBZ filter's cd_values."""
    version = cd_values[0] if len(cd_values) > 0 else 0
    int_size = cd_values[1] if len(cd_values) > 1 else 0
    zigzag = cd_values[2] if len(cd_values) > 2 else 0
    zstd_level = cd_values[3] if len(cd_values) > 3 else 1
    return version, int_size, zigzag, zstd_level


def _vbz_body(chunk: bytes, int_size: int, zstd_level: int):
    """A VBZ chunk's sample count and its StreamVByte body (zstd undone)."""
    if len(chunk) < 4:
        raise Fast5FormatError('VBZ: chunk shorter than its size header')
    (orig_size,) = struct.unpack_from('<I', chunk, 0)
    n = orig_size // int_size
    body = chunk[4:]
    if zstd_level:
        body = zstd_decompress(body, n * 5 + 16)
    return n, body


def vbz_decode_body(body: bytes, n: int, version: int, int_size: int, zigzag: int) -> bytes:
    """StreamVByte body of ``n`` integers (after zstd) -> raw little-endian integers."""
    buf = np.frombuffer(body, dtype=np.uint8)
    if int_size in (1,):
        raise Fast5FormatError('VBZ: 1-byte integers are not used by fast5 signals')
    if version == 0 or int_size == 4:
        u = _svb_decode_u32(buf, n)
        if zigzag:
            d = (u >> np.uint32(1)).astype(np.int32) ^ -(u & np.uint32(1)).astype(np.int32)
            vals = np.cumsum(d, dtype=np.int64)
        else:
            vals = u.astype(np.int64)
    elif version == 1 and int_size == 2:
        u = _svb_decode_u16(buf, n)
        if zigzag:
            d = (u >> np.uint16(1)).astype(np.int16) ^ -(u & np.uint16(1)).astype(np.int16)
            vals = np.cumsum(d.astype(np.int64))
        else:
            vals = u.astype(np.int64)
    else:
        raise Fast5FormatError(f'VBZ: unsupported version {version} / integer size {int_size}')
    dt = {2: '<i2', 4: '<i4'}[int_size] if zigzag else {2: '<u2', 4: '<u4'}[int_size]
    return vals.astype(dt).tobytes()


def vbz_decompress(chunk: bytes, cd_values: Tuple[int, ...]) -> bytes:
    """One HDF5 chunk written by the VBZ filter -> raw little-endian integers."""
    version, int_size, zigzag, zstd_level = _vbz_params(cd_values)
    if int_size == 0:                                   # bytes passed through zstd only
        if len(chunk) < 4:
            raise Fast5FormatError('VBZ: chunk shorter than its size header')
        (orig_size,) = struct.unpack_from('<I', chunk, 0)
        body = chunk[4:]
        return zstd_decompress(body, orig_size) if zstd_level else bytes(body[:orig_size])
    n, body = _vbz_body(chunk, int_size, zstd_level)
    return vbz_decode_body(body, n, version, int_size, zigzag)


def zstd_frame_size(frame: bytes, max_size: int) -> int:
    """Frame_Content_Size of ``frame`` if the device decoder (wstr_zstd_decode_batch) can take it, else -1.
    Decided from the bytes alone by walking the frame header and the 3-byte block headers: exactly one
    frame, ending at the payload's end, no dictionary ID, no content checksum, a content size present and
    at most ``max_size`` (the bound the host decoder uses).  Anything else is decoded on the host."""
    n = len(frame)
    if n < 9 or frame[:4] != b'\x28\xb5\x2f\xfd':
        return -1
    fhd = frame[4]
    single, fcs_id = (fhd >> 5) & 1, fhd >> 6
    if fhd & 0x0F:                                  # reserved bit, content checksum or dictionary ID
        return -1
    if not single and (frame[5] >> 3) + 10 > 31:
        return -1
    p = 5 + (not single)
    width = (0, 2, 4, 8)[fcs_id] or (1 if single else 0)
    if width == 0 or p + width + 3 > n:
        return -1
    fcs = int.from_bytes(frame[p:p + width], 'little') + (256 if width == 2 else 0)
    if fcs > max_size:
        return -1
    p += width
    while True:
        if p + 3 > n:
            return -1
        h = int.from_bytes(frame[p:p + 3], 'little')
        p += 3
        btype, size = (h >> 1) & 3, h >> 3
        if btype == 3 or (btype == 2 and size > 1 << 17):
            return -1
        p += 1 if btype == 1 else size
        if p > n:
            return -1
        if h & 1:
            return fcs if p == n else -1


# chunk kinds of stored_chunks / raw_chunks: 0-2 are the numbering of wstr_vbz_decode_batch, and a VBZ chunk
# whose payload is still its zstd frame (for wstr_zstd_decode_batch, then the StreamVByte decode) is 3 or 4
KIND_VBZ0, KIND_VBZ1, KIND_RAW, KIND_VBZ0_ZSTD, KIND_VBZ1_ZSTD = 0, 1, 2, 3, 4


class RawChunk(NamedTuple):
    """One chunk of a read's signal as the device decoder takes it: samples [start, start + count) of the
    read come from ``payload`` -- a VBZ StreamVByte body after zstd (kind KIND_VBZ0 / KIND_VBZ1, coding
    ``coded`` >= count samples, zig-zag deltas if ``zigzag``), the zstd frame of such a body (KIND_VBZ0_ZSTD /
    KIND_VBZ1_ZSTD, ``body_size`` its Frame_Content_Size) or ``count`` little-endian int16 (KIND_RAW)."""
    start: int
    count: int
    kind: int
    payload: bytes
    zigzag: bool = False
    coded: int = 0
    body_size: int = 0

    def unzstd(self) -> 'RawChunk':
        """The chunk with its zstd frame (if any) undone on the host."""
        if self.kind < KIND_VBZ0_ZSTD:
            return self
        body = zstd_decompress(self.payload, self.coded * 5 + 16)
        return self._replace(kind=self.kind - KIND_VBZ0_ZSTD, payload=body, body_size=0)

    def decode(self) -> np.ndarray:
        """The chunk's int16 samples, decoded on the host (fast5.vbz_decompress)."""
        c = self.unzstd()
        if c.kind == KIND_RAW:
            return np.frombuffer(c.payload, dtype='<i2', count=c.count)
        raw = vbz_decode_body(c.payload, c.coded, c.kind, 2, int(c.zigzag))
        return np.frombuffer(raw, dtype='<i2', count=c.count)


@dataclass
class CompressedRead:
    """A read's raw signal as its file stores it (see ``raw_chunks``)."""
    path: str
    read_name: Optional[str]
    n_samples: int
    chunks: List[RawChunk]

    def decode(self) -> np.ndarray:
        """The read's int16 samples decoded on the host: what ``raw_signal`` returns."""
        out = np.zeros(self.n_samples, dtype=np.int16)
        for c in self.chunks:
            out[c.start:c.start + c.count] = c.decode()
        return out


def _unshuffle(data: bytes, elem: int) -> bytes:
    n = len(data) // elem
    a = np.frombuffer(data[:n * elem], dtype=np.uint8).reshape(elem, n)
    return a.T.tobytes() + data[n * elem:]


# ---------------------------------------------------------------------------------------------------
# HDF5
# ---------------------------------------------------------------------------------------------------
class _Obj:
    """Parsed object header: the messages this reader cares about."""

    def __init__(self):
        self.symtab = None          # (btree address, heap address)
        self.links = {}             # compact new-style links: name -> object header address
        self.dense_links = False    # links kept in a fractal heap (not supported)
        self.shape = None
        self.dtype = None
        self.layout = None          # ('contiguous', addr, size) | ('compact', bytes) | ('chunked', btree, chunk dims)
        self.filters = []           # [(id, cd_values)]


class H5File:
    def __init__(self, path: str):
        self.path = path
        self._fh = open(path, 'rb')
        try:
            self.buf = mmap.mmap(self._fh.fileno(), 0, access=mmap.ACCESS_READ)
        except ValueError as exc:
            self._fh.close()
            raise Fast5FormatError(f'{path}: empty file') from exc
        b = self.buf
        if b[:8] != b'\x89HDF\r\n\x1a\n':
            raise Fast5FormatError(f'{path}: not an HDF5 file')
        if b[8] not in (0, 1):
            raise Fast5FormatError(f'{path}: HDF5 superblock version {b[8]} is not supported (only 0/1)')
        if b[13] != 8 or b[14] != 8:
            raise Fast5FormatError(f'{path}: only 8-byte offsets and lengths are supported')
        pos = 24 + (4 if b[8] == 1 else 0)
        self.base = struct.unpack_from('<Q', b, pos)[0]
        entry = pos + 32
        _, ohdr, cache, _ = struct.unpack_from('<QQII', b, entry)
        self._objs: Dict[int, _Obj] = {}
        self._groups: Dict[int, Dict[str, int]] = {}
        self.root = ohdr

    def close(self):
        try:
            self.buf.close()
        finally:
            self._fh.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # -- object headers (version 1) ---------------------------------------------------------------
    def _object(self, addr: int) -> _Obj:
        if addr in self._objs:
            return self._objs[addr]
        b = self.buf
        a = addr + self.base
        if b[a:a + 4] == b'OHDR':
            raise Fast5FormatError(f'{self.path}: version-2 object headers are not supported')
        version, _, nmsg, _, hsize = struct.unpack_from('<BBHII', b, a)
        if version != 1:
            raise Fast5FormatError(f'{self.path}: bad object header at {addr}')
        obj = _Obj()
        blocks = [(a + 16, hsize)]
        seen = 0
        while blocks and seen < nmsg:
            p, size = blocks.pop(0)
            end = p + size
            while p + 8 <= end and seen < nmsg:
                mtype, msize, _flags = struct.unpack_from('<HHB', b, p)
                body = p + 8
                self._message(obj, mtype, body, msize, blocks)
                p = body + msize
                seen += 1
        self._objs[addr] = obj
        return obj

    def _message(self, obj: _Obj, mtype: int, p: int, size: int, blocks: List[Tuple[int, int]]):
        b = self.buf
        if mtype == 0x0010:                                   # continuation
            off, ln = struct.unpack_from('<QQ', b, p)
            blocks.append((off + self.base, ln))
        elif mtype == 0x0011:                                 # symbol table (old-style group)
            obj.symtab = struct.unpack_from('<QQ', b, p)
        elif mtype == 0x0006:                                 # link message (compact new-style group)
            flags = b[p + 1]
            q = p + 2
            ltype = 0
            if flags & 0x08:
                ltype = b[q]
                q += 1
            if flags & 0x04:
                q += 8
            if flags & 0x10:
                q += 1
            nsz = 1 << (flags & 3)
            nlen = int.from_bytes(b[q:q + nsz], 'little')
            q += nsz
            name = bytes(b[q:q + nlen]).decode('utf-8', 'replace')
            q += nlen
            if ltype == 0:                                    # hard link
                (obj.links[name],) = struct.unpack_from('<Q', b, q)
        elif mtype == 0x0002:                                 # link info: is there a fractal heap?
            flags = b[p + 1]
            q = p + 2 + (8 if flags & 1 else 0)
            (fheap,) = struct.unpack_from('<Q', b, q)
            obj.dense_links = fheap != UNDEF
        elif mtype == 0x0001:                                 # dataspace
            ver, rank, flags = struct.unpack_from('<BBB', b, p)
            q = p + (8 if ver == 1 else 4)
            obj.shape = struct.unpack_from('<%dQ' % rank, b, q) if rank else ()
        elif mtype == 0x0003:                                 # datatype: fixed-point only
            cv, bits0, _, _, tsize = struct.unpack_from('<BBBBI', b, p)
            cls = cv & 0x0f
            if cls == 0:
                signed = bool(bits0 & 0x08)
                big = bool(bits0 & 0x01)
                obj.dtype = np.dtype(('>' if big else '<') + ('i' if signed else 'u') + str(tsize))
            else:
                obj.dtype = ('class', cls, tsize)
        elif mtype == 0x0008:                                 # data layout
            ver = b[p]
            if ver == 3:
                cls = b[p + 1]
                if cls == 0:
                    (n,) = struct.unpack_from('<H', b, p + 2)
                    obj.layout = ('compact', bytes(b[p + 4:p + 4 + n]))
                elif cls == 1:
                    addr, n = struct.unpack_from('<QQ', b, p + 2)
                    obj.layout = ('contiguous', addr, n)
                elif cls == 2:
                    nd = b[p + 2]
                    (bt,) = struct.unpack_from('<Q', b, p + 3)
                    dims = struct.unpack_from('<%dI' % nd, b, p + 11)
                    obj.layout = ('chunked', bt, dims)
            elif ver in (1, 2):
                nd, cls = b[p + 1], b[p + 2]
                q = p + 8
                addr = None
                if cls != 0:
                    (addr,) = struct.unpack_from('<Q', b, q)
                    q += 8
                dims = struct.unpack_from('<%dI' % nd, b, q)
                q += 4 * nd
                if cls == 1:
                    obj.layout = ('contiguous', addr, None)
                elif cls == 2:
                    obj.layout = ('chunked', addr, dims)
                else:
                    (n,) = struct.unpack_from('<I', b, q)
                    obj.layout = ('compact', bytes(b[q + 4:q + 4 + n]))
            else:
                raise Fast5FormatError(f'{self.path}: data layout message version {ver} is not supported')
        elif mtype == 0x000B:                                 # filter pipeline
            ver, nf = b[p], b[p + 1]
            q = p + (8 if ver == 1 else 2)
            for _ in range(nf):
                (fid,) = struct.unpack_from('<H', b, q)
                q += 2
                name_len = 0
                if ver == 1 or fid >= 256:
                    (name_len,) = struct.unpack_from('<H', b, q)
                    q += 2
                _fl, ncd = struct.unpack_from('<HH', b, q)
                q += 4
                if ver == 1:
                    name_len = (name_len + 7) // 8 * 8
                q += name_len
                cd = struct.unpack_from('<%dI' % ncd, b, q)
                q += 4 * ncd
                if ver == 1 and ncd % 2:
                    q += 4
                obj.filters.append((fid, cd))

    # -- groups -----------------------------------------------------------------------------------
    def _members(self, addr: int) -> Dict[str, int]:
        if addr in self._groups:
            return self._groups[addr]
        obj = self._object(addr)
        if obj.dense_links:
            raise Fast5FormatError(f'{self.path}: groups with fractal-heap link storage are not supported')
        if obj.symtab is None:
            if obj.links or obj.layout is None:
                self._groups[addr] = dict(obj.links)
                return self._groups[addr]
            raise Fast5FormatError(f'{self.path}: object at {addr} is not a group')
        bt, heap = obj.symtab
        b = self.buf
        h = heap + self.base
        if b[h:h + 4] != b'HEAP':
            raise Fast5FormatError(f'{self.path}: bad local heap')
        (data_addr,) = struct.unpack_from('<Q', b, h + 24)
        data_addr += self.base
        out: Dict[str, int] = {}

        def walk(node):
            n = node + self.base
            sig = b[n:n + 4]
            if sig == b'TREE':
                ntype, _level, used = struct.unpack_from('<BBH', b, n + 4)
                if ntype != 0:
                    raise Fast5FormatError(f'{self.path}: group B-tree expected')
                p = n + 24 + 8                          # skip key 0
                for _ in range(used):
                    (child,) = struct.unpack_from('<Q', b, p)
                    walk(child)
                    p += 16                             # child + next key
            elif sig == b'SNOD':
                (nsym,) = struct.unpack_from('<H', b, n + 6)
                p = n + 8
                for _ in range(nsym):
                    name_off, ohdr = struct.unpack_from('<QQ', b, p)
                    s = data_addr + name_off
                    e = b.find(b'\x00', s)
                    out[b[s:e].decode('utf-8', 'replace')] = ohdr
                    p += 40
            else:
                raise Fast5FormatError(f'{self.path}: bad group node')

        if bt != UNDEF:
            walk(bt)
        out.update(obj.links)
        self._groups[addr] = out
        return out

    def keys(self, path: str = '/') -> List[str]:
        return sorted(self._members(self._resolve(path)))

    def _resolve(self, path: str) -> int:
        addr = self.root
        for part in [p for p in path.split('/') if p]:
            members = self._members(addr)
            if part not in members:
                raise KeyError(f'{path} not found in {self.path}')
            addr = members[part]
        return addr

    def __contains__(self, path: str) -> bool:
        try:
            self._resolve(path)
            return True
        except (KeyError, Fast5FormatError):
            return False

    # -- datasets ---------------------------------------------------------------------------------
    def dataset(self, path: str) -> np.ndarray:
        obj = self._object(self._resolve(path))
        if obj.layout is None or obj.shape is None or not isinstance(obj.dtype, np.dtype):
            raise Fast5FormatError(f'{path}: not an integer dataset this reader understands')
        shape = tuple(int(d) for d in obj.shape)
        count = int(np.prod(shape)) if shape else 1
        elem = obj.dtype.itemsize
        kind = obj.layout[0]
        b = self.buf
        if kind == 'compact':
            raw = obj.layout[1]
        elif kind == 'contiguous':
            addr = obj.layout[1]
            raw = b'' if addr == UNDEF else bytes(b[addr + self.base:addr + self.base + count * elem])
        else:
            if len(shape) != 1:
                raise Fast5FormatError(f'{path}: only one-dimensional chunked datasets are supported')
            raw = self._read_chunks(obj, shape[0], elem)
        arr = np.frombuffer(raw, dtype=obj.dtype, count=count)
        return arr.reshape(shape).astype(obj.dtype.newbyteorder('='), copy=True)

    def _chunk_entries(self, obj: _Obj) -> Iterator[Tuple[int, int, int, int]]:
        """(first element, stored bytes, filter mask, address) of every chunk in the v1 chunk B-tree."""
        _, bt, dims = obj.layout
        b = self.buf
        nd = len(dims)
        key_size = 8 + 8 * nd

        def walk(node):
            p = node + self.base
            if b[p:p + 4] != b'TREE':
                raise Fast5FormatError(f'{self.path}: bad chunk B-tree')
            ntype, level, used = struct.unpack_from('<BBH', b, p + 4)
            if ntype != 1:
                raise Fast5FormatError(f'{self.path}: chunk B-tree expected')
            q = p + 24
            for _ in range(used):
                csize, fmask = struct.unpack_from('<II', b, q)
                offs = struct.unpack_from('<%dQ' % nd, b, q + 8)
                (child,) = struct.unpack_from('<Q', b, q + key_size)
                if level > 0:
                    yield from walk(child)
                else:
                    yield int(offs[0]), csize, fmask, child
                q += key_size + 8

        if bt != UNDEF:
            yield from walk(bt)

    def _chunk_bytes(self, addr: int, csize: int) -> bytes:
        return bytes(self.buf[addr + self.base:addr + self.base + csize])

    def _unfilter(self, obj: _Obj, data: bytes, fmask: int, elem: int) -> bytes:
        for idx in range(len(obj.filters) - 1, -1, -1):
            if fmask & (1 << idx):
                continue
            fid, cd = obj.filters[idx]
            if fid == VBZ_FILTER_ID:
                data = vbz_decompress(data, cd)
            elif fid == 1:
                data = zlib.decompress(data)
            elif fid == 2:
                data = _unshuffle(data, elem)
            elif fid == 3:
                data = data[:-4]              # fletcher32 checksum, not verified
            else:
                raise Fast5FormatError(f'{self.path}: HDF5 filter {fid} is not supported')
        return data

    def _read_chunks(self, obj: _Obj, n: int, elem: int) -> bytes:
        chunk_elems = int(obj.layout[2][0])
        out = bytearray(n * elem)
        for start, csize, fmask, addr in self._chunk_entries(obj):
            data = self._unfilter(obj, self._chunk_bytes(addr, csize), fmask, elem)
            take = min(chunk_elems, n - start) * elem
            if take > 0:
                if len(data) < take:
                    raise Fast5FormatError(f'{self.path}: chunk shorter than its extent')
                out[start * elem:start * elem + take] = data[:take]
        return bytes(out)

    def raw_chunks(self, path: str) -> Tuple[int, List[RawChunk]]:
        """An int16 signal dataset as (sample count, chunks covering [0, count) in order) without the
        StreamVByte decode: a VBZ chunk of 2-byte integers comes back as its body after zstd (kind KIND_VBZ0
        or KIND_VBZ1); every other chunk -- other filters, other VBZ integer sizes, contiguous and compact
        layouts -- is decoded here, as ``dataset`` decodes it, and comes back verbatim (KIND_RAW), and so
        do unallocated chunks (zeros, as ``dataset`` leaves them)."""
        return self._chunks(path, keep_frames=False)

    def stored_chunks(self, path: str) -> Tuple[int, List[RawChunk]]:
        """``raw_chunks`` with VBZ chunks as the file stores them: a chunk whose zstd frame the device decoder
        takes (``zstd_frame_size``) comes back as that frame (KIND_VBZ0_ZSTD / KIND_VBZ1_ZSTD); any other zstd
        frame is undone here."""
        return self._chunks(path, keep_frames=True)

    # -- reads (the interface fast5.open_raw's readers share with pod5.Pod5File) ------------------------------
    def read_names(self) -> List[str]:
        """Read ids of a multi-read fast5 (group names ``read_<id>``)."""
        return [k[5:] for k in self.keys('/') if k.startswith('read_')]

    def read_signal(self, read_name: Optional[str]) -> np.ndarray:
        return _raw_signal(self, read_name)

    def read_chunks(self, read_name: Optional[str], keep_frames: bool) -> 'CompressedRead':
        """The read's signal dataset as ``stored_chunks`` (``keep_frames``) or ``raw_chunks`` returns it."""
        n, chunks = self._chunks(_signal_path(self, read_name), keep_frames)
        return CompressedRead(self.path, read_name, n, chunks)

    def _chunks(self, path: str, keep_frames: bool) -> Tuple[int, List[RawChunk]]:
        obj = self._object(self._resolve(path))
        vbz = None
        if (obj.layout is not None and obj.layout[0] == 'chunked' and obj.shape is not None and len(obj.shape) == 1
                and obj.dtype == np.dtype('<i2') and len(obj.filters) == 1 and obj.filters[0][0] == VBZ_FILTER_ID):
            version, int_size, zigzag, zstd_level = _vbz_params(obj.filters[0][1])
            if int_size == 2 and version in (0, 1):
                vbz = version, zigzag, zstd_level
        if vbz is None:
            x = np.ascontiguousarray(self.dataset(path), dtype=np.int16).reshape(-1)
            return len(x), [RawChunk(0, len(x), KIND_RAW, x.tobytes())]
        version, zigzag, zstd_level = vbz
        n = int(obj.shape[0])
        chunk_elems = int(obj.layout[2][0])
        found = []
        for start, csize, fmask, addr in self._chunk_entries(obj):
            take = min(chunk_elems, n - start)
            if take <= 0:
                continue
            data = self._chunk_bytes(addr, csize)
            if fmask & 1:                                       # stored without the filter
                data = self._unfilter(obj, data, fmask, 2)
                if len(data) < 2 * take:
                    raise Fast5FormatError(f'{self.path}: chunk shorter than its extent')
                found.append(RawChunk(start, take, KIND_RAW, data[:2 * take]))
                continue
            kind = KIND_VBZ0 if version == 0 else KIND_VBZ1
            size = -1
            if keep_frames and zstd_level and len(data) >= 4:
                coded = struct.unpack_from('<I', data, 0)[0] // 2
                size = zstd_frame_size(data[4:], coded * 5 + 16)
            if size >= 0:
                body, kind = data[4:], kind + KIND_VBZ0_ZSTD
            else:
                coded, body = _vbz_body(data, 2, zstd_level)
            if coded < take:
                raise Fast5FormatError(f'{self.path}: chunk shorter than its extent')
            found.append(RawChunk(start, take, kind, body, bool(zigzag), coded, max(size, 0)))
        found.sort(key=lambda c: c.start)
        chunks, at = [], 0
        for c in found:
            if c.start < at:
                raise Fast5FormatError(f'{self.path}: overlapping chunks')
            if c.start > at:
                chunks.append(RawChunk(at, c.start - at, KIND_RAW, bytes(2 * (c.start - at))))
            chunks.append(c)
            at = c.start + c.count
        if at < n:
            chunks.append(RawChunk(at, n - at, KIND_RAW, bytes(2 * (n - at))))
        return n, chunks


# ---------------------------------------------------------------------------------------------------
# fast5 and POD5: one entry point per question, the container chosen from the file's first bytes
# ---------------------------------------------------------------------------------------------------
HDF5_SIGNATURE = b'\x89HDF\r\n\x1a\n'
POD5_SIGNATURE = b'\x8bPOD\r\n\x1a\n'


def open_raw(path: str):
    """The raw-signal file at ``path``, opened with the reader its first 8 bytes name: an ``H5File`` for fast5
    (HDF5), a ``pod5.Pod5File`` for POD5.  Both answer ``read_names()``, ``read_signal(read_name)`` and
    ``read_chunks(read_name, keep_frames)`` and are context managers, so no caller looks at the file type."""
    with open(path, 'rb') as fh:
        head = fh.read(8)
    if head == POD5_SIGNATURE:
        from . import pod5
        return pod5.Pod5File(path)
    return H5File(path)                 # HDF5; anything else gets H5File's own 'not an HDF5 file' or 'empty file'


def read_names(path: str) -> List[str]:
    """Read ids of a multi-read fast5 (group names ``read_<id>``) or of a POD5 file."""
    with open_raw(path) as f:
        return f.read_names()


def raw_signal(path: str, read_name: Optional[str] = None) -> np.ndarray:
    """The raw int16 DAC samples of one read.  ``read_name`` selects a read of a multi-read
    fast5 or a POD5 file; a single-read file (``Raw/Reads/Read_<n>``) has only one."""
    with open_raw(path) as f:
        return f.read_signal(read_name)


def _raw_signal(h5: H5File, read_name: Optional[str]) -> np.ndarray:
    return h5.dataset(_signal_path(h5, read_name))


def _signal_path(h5: H5File, read_name: Optional[str]) -> str:
    """The dataset holding a read's signal: ``read_<name>/Raw/Signal`` (the ``read_`` prefix optional),
    else the first read of a single-read file, else the only read of a multi-read file."""
    if read_name is not None:
        name = read_name if read_name.startswith('read_') else 'read_' + read_name
        if name in h5:
            return f'{name}/Raw/Signal'
    if 'Raw/Reads' in h5:
        reads = h5.keys('Raw/Reads')
        if reads:
            return f'Raw/Reads/{reads[0]}/Signal'         # fast5.py:50-52: the first read
    if read_name is None:
        members = [k for k in h5.keys('/') if k.startswith('read_')]
        if len(members) == 1:
            return f'{members[0]}/Raw/Signal'
    raise KeyError(f'read {read_name} not found in {h5.path}')


def raw_chunks(path: str, read_name: Optional[str] = None, h5=None) -> CompressedRead:
    """One read's signal as its file stores it, for the device decoder (CallerEngine.call_vbz_batch):
    the read is chosen exactly as ``raw_signal`` chooses it, zstd is undone here and the StreamVByte
    decode is left to the GPU (see H5File.raw_chunks; a POD5 signal row is one chunk, see pod5.py).
    ``h5``: the file, already open (``open_raw``)."""
    if h5 is None:
        with open_raw(path) as f:
            return f.read_chunks(read_name, False)
    return h5.read_chunks(read_name, False)


def stored_chunks(path: str, read_name: Optional[str] = None, h5=None) -> CompressedRead:
    """``raw_chunks`` with the zstd frames the device decodes left as the file stores them (see
    H5File.stored_chunks): the read's chunks cross PCIe as stored and zstd is undone on the GPU too."""
    if h5 is None:
        with open_raw(path) as f:
            return f.read_chunks(read_name, True)
    return h5.read_chunks(read_name, True)


class Fast5:
    """The reference's ``Fast5(path, get_data_only=True)`` (schemas/fast5.py:9-57): raw data,
    spike removal, MAD normalisation, window slice -- the last three on the GPU."""

    def __init__(self, fast5path: str, get_data_only: bool = True, read_name: Optional[str] = None,
                 spike_removal: str = 'Brute'):
        if not get_data_only:
            raise NotImplementedError('basecall tables (Analyses/...) are outside the caller path')
        self.path = fast5path
        self.read_name = read_name
        self.spike_removal = spike_removal
        self.data: Optional[np.ndarray] = None
        self.norm: Optional[np.ndarray] = None

    def get_raw(self) -> np.ndarray:
        if self.data is None:
            self.data = np.ascontiguousarray(raw_signal(self.path, self.read_name), dtype=np.int16)
        return self.data

    def get_data_processed(self, position: Optional[Tuple[int, int]] = None) -> np.ndarray:
        from .normalize import get_data_processed
        return get_data_processed(self.get_raw(), position, self.spike_removal)
