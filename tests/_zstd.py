"""libzstd through ctypes for the zstd tests: compression with chosen frame parameters, the reference decode
the device decoder is held to, and the corpus of frames it is checked on."""
import ctypes

import numpy as np

import _h5write as hw
from warpstr_b200 import fast5, synth

C_LEVEL, C_WINDOW_LOG, C_CONTENT_SIZE, C_CHECKSUM = 100, 101, 200, 201
UNKNOWN = 2 ** 64 - 1


def lib():
    z = fast5._libzstd()
    z.ZSTD_createCCtx.restype = ctypes.c_void_p
    z.ZSTD_freeCCtx.argtypes = [ctypes.c_void_p]
    z.ZSTD_CCtx_setParameter.restype = ctypes.c_size_t
    z.ZSTD_CCtx_setParameter.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int]
    z.ZSTD_compress2.restype = ctypes.c_size_t
    z.ZSTD_compress2.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t]
    z.ZSTD_compressBound.restype = ctypes.c_size_t
    z.ZSTD_compressBound.argtypes = [ctypes.c_size_t]
    return z


def compress(data: bytes, level: int = 1, checksum: bool = False, content_size: bool = True,
             window_log: int = 0) -> bytes:
    z = lib()
    cctx = z.ZSTD_createCCtx()
    try:
        for p, v in ((C_LEVEL, level), (C_CHECKSUM, int(checksum)), (C_CONTENT_SIZE, int(content_size)),
                     (C_WINDOW_LOG, window_log)):
            assert not z.ZSTD_isError(z.ZSTD_CCtx_setParameter(cctx, p, v))
        cap = z.ZSTD_compressBound(len(data))
        out = ctypes.create_string_buffer(max(cap, 1))
        n = z.ZSTD_compress2(cctx, out, cap, data, len(data))
        assert not z.ZSTD_isError(n)
        return out.raw[:n]
    finally:
        z.ZSTD_freeCCtx(cctx)


def version() -> int:
    """libzstd's ZSTD_versionNumber (10505 for 1.5.5)."""
    return int(lib().ZSTD_versionNumber())


def content_size(frame: bytes) -> int:
    """Frame_Content_Size as libzstd reads it; -1 when the header has none or is not a frame's."""
    n = lib().ZSTD_getFrameContentSize(frame, len(frame))
    return -1 if n >= 2 ** 64 - 2 else int(n)


def reference(frame: bytes, size: int):
    """What the device must produce for ``frame`` told it holds ``size`` bytes: libzstd's output when libzstd
    decodes the frame, with that content size in its header, to exactly that many bytes; else None."""
    if content_size(frame) != size:
        return None
    z = lib()
    out = ctypes.create_string_buffer(max(size, 1))
    got = z.ZSTD_decompress(out, size, frame, len(frame))
    if z.ZSTD_isError(got) or got != size:
        return None
    return out.raw[:size]


def synthetic_raw(n: int, seed: int = 0) -> np.ndarray:
    """int16 samples of synthetic HD reads (synth.to_raw_int16), concatenated to ``n``."""
    rng = np.random.default_rng(seed)
    locus = synth.make_locus('HD', seed=seed)
    parts, have = [], 0
    k = 0
    while have < n:
        for r in synth.make_reads(locus, 4, seed=seed * 100 + k):
            raw, _, _ = synth.to_raw_int16(rng, r.signal, pad=4096)
            parts.append(raw)
            have += len(raw)
        k += 1
    return np.concatenate(parts)[:n].astype(np.int16)


def vbz_bodies(n_chunks: int = 2, samples: int = 102400, seed: int = 0):
    """(name, body) of VBZ v0 and v1 StreamVByte bodies of synthetic reads, ``samples`` per chunk."""
    x = synthetic_raw(n_chunks * samples, seed)
    out = []
    for v in (0, 1):
        for c in range(n_chunks):
            out.append((f'vbz{v}-{c}', hw.svb_body(x[c * samples:(c + 1) * samples], v)))
    return out


def plain_data(seed: int = 0):
    """(name, bytes): random, constant, periodic (periods 1-31), long-range repeats and the FCS-field edges."""
    rng = np.random.default_rng(seed)
    out = [('random', rng.integers(0, 256, 50000, dtype=np.uint8).tobytes()),
           ('constant', bytes([7]) * 70000), ('empty-ish', b'a')]
    for p in range(1, 32):
        unit = rng.integers(0, 256, p, dtype=np.uint8).tobytes()
        out.append((f'period{p}', (unit * (3000 // p + 2))[:3000 + p]))
    block = rng.integers(0, 256, 20000, dtype=np.uint8).tobytes()
    noise = rng.integers(0, 4, 200000, dtype=np.uint8)
    far = np.frombuffer(block * 10, dtype=np.uint8)[:200000] ^ (noise == 0).astype(np.uint8)
    out.append(('long-range', far.tobytes()))
    text = b' '.join(rng.choice([b'alpha', b'beta', b'gamma', b'delta', b'eps'], 60000))
    out.append(('words', text))
    # multi-block: treeless literals and repeated tables (copies), RLE blocks (const), RLE tables (sparse)
    words = [b'alpha', b'beta', b'gamma', b'delta', b'eps', b'zeta', b'eta', b'theta']
    text = b' '.join(rng.choice(words, 30000))
    parts = [text[:130000]]
    for _ in range(60):
        a = int(rng.integers(0, 100000))
        parts.append(text[a:a + 3000] + bytes(rng.choice(list(b'abdeghlmpt'), 40)))
    out.append(('copies', b''.join(parts)))
    out.append(('const-long', bytes([9]) * 300000))
    sparse = bytearray(b'A' * 200000)
    sparse[::997] = b'B' * len(sparse[::997])
    out.append(('sparse', bytes(sparse)))
    for n in (1, 255, 256, 65791, 65792):
        out.append((f'fcs{n}', (rng.integers(0, 16, n, dtype=np.uint8) * 3).tobytes()))
    return out


LEVELS = (-5, 1, 3, 9, 19)


def corpus(seed: int = 0):
    """(name, frame, content) of every frame the device decoder is checked on."""
    out = []
    for name, body in vbz_bodies(seed=seed):
        for lv in LEVELS:
            out.append((f'{name}-L{lv}', compress(body, lv), body))
    for name, data in plain_data(seed):
        for lv in (1, 19):
            out.append((f'{name}-L{lv}', compress(data, lv), data))
    return out


def hand_frames():
    """(name, frame, content) of frames no libzstd level writes: a compressed block with RLE literals and RLE
    tables for LL, OF and ML (4 literals 'A', then one sequence: offset 1, match length 10)."""
    block = bytes([(4 << 3) | 1, 0x41,            # literals: RLE, 4 x 'A'
                   1, 0x54,                       # one sequence; LL, OF, ML tables all RLE
                   4, 2, 7,                       # LL code 4 (4), OF code 2 (offset 1 + 2 bits), ML code 7 (10)
                   0x04])                         # bitstream: the offset's 2 bits (0) under the end mark
    hdr = (len(block) << 3) | (2 << 1) | 1
    frame = (0xFD2FB528).to_bytes(4, 'little') + bytes([0x20, 14]) + hdr.to_bytes(3, 'little') + block
    return [('rle-literals', frame, b'A' * 14)]
