"""CPU: the fast5 reader (warpstr_b200/fast5.py) -- VBZ decoding against an encoder written here
from the published format, and the refusal of files that are not HDF5."""
import ctypes
import struct

import numpy as np
import pytest

from warpstr_b200 import fast5


def _zstd_compress(data: bytes) -> bytes:
    lib = fast5._libzstd()
    lib.ZSTD_compressBound.restype = ctypes.c_size_t
    lib.ZSTD_compressBound.argtypes = [ctypes.c_size_t]
    lib.ZSTD_compress.restype = ctypes.c_size_t
    lib.ZSTD_compress.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int]
    cap = lib.ZSTD_compressBound(len(data))
    out = ctypes.create_string_buffer(cap)
    n = lib.ZSTD_compress(out, cap, data, len(data), 1)
    assert not lib.ZSTD_isError(n)
    return out.raw[:n]


def _vbz_encode(x: np.ndarray, version: int, zstd: bool = True) -> bytes:
    """int16 samples -> one VBZ chunk: zig-zag of the deltas, StreamVByte (32-bit codes in
    version 0, the 16-bit variant in version 1), optional zstd, uint32 byte-size header."""
    x = x.astype(np.int64)
    d = np.diff(x, prepend=0)
    if version == 0:
        zz = ((d << 1) ^ (d >> 31)) & 0xFFFFFFFF
        ctrl = bytearray((len(x) + 3) // 4)
        data = bytearray()
        for i, v in enumerate(zz.tolist()):
            nb = 1 if v < 1 << 8 else 2 if v < 1 << 16 else 3 if v < 1 << 24 else 4
            ctrl[i >> 2] |= (nb - 1) << (2 * (i & 3))
            data += int(v).to_bytes(nb, 'little')
    else:
        d = ((d + 32768) % 65536) - 32768      # 16-bit arithmetic wraps
        zz = ((d << 1) ^ (d >> 15)) & 0xFFFF
        ctrl = bytearray((len(x) + 7) // 8)
        data = bytearray()
        for i, v in enumerate(zz.tolist()):
            nb = 1 if v < 1 << 8 else 2
            ctrl[i >> 3] |= (nb - 1) << (i & 7)
            data += int(v).to_bytes(nb, 'little')
    body = bytes(ctrl) + bytes(data)
    if zstd:
        body = _zstd_compress(body)
    return struct.pack('<I', 2 * len(x)) + body


@pytest.mark.parametrize('version', [0, 1])
@pytest.mark.parametrize('n', [0, 1, 3, 4, 5, 8, 9, 1000, 4097])
def test_vbz_round_trip(version, n):
    rng = np.random.default_rng(100 * version + n)
    x = (450 + np.cumsum(rng.integers(-40, 41, size=n))).astype(np.int16)
    if n > 10:
        x[7] = 32767          # extreme jumps need the wide codes
        x[8] = -32768
    for zstd in (True, False):
        chunk = _vbz_encode(x, version, zstd)
        raw = fast5.vbz_decompress(chunk, (version, 2, 1, 1 if zstd else 0))
        assert np.array_equal(np.frombuffer(raw, dtype='<i2'), x)


def test_vbz_rejects_truncated_chunk():
    x = np.arange(100, dtype=np.int16)
    chunk = _vbz_encode(x, 0, zstd=False)
    with pytest.raises(fast5.Fast5FormatError):
        fast5.vbz_decompress(chunk[:-5], (0, 2, 1, 0))
    with pytest.raises(fast5.Fast5FormatError):
        fast5.vbz_decompress(b'\x01', (0, 2, 1, 0))


def test_not_hdf5(tmp_path):
    p = tmp_path / 'x.fast5'
    p.write_bytes(b'not an hdf5 file at all')
    with pytest.raises(fast5.Fast5FormatError):
        fast5.H5File(str(p))
    (tmp_path / 'empty.fast5').write_bytes(b'')
    with pytest.raises(fast5.Fast5FormatError):
        fast5.H5File(str(tmp_path / 'empty.fast5'))
