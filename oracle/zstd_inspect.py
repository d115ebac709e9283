"""Header-level inspector of a zstd frame (RFC 8878): what each block uses, read from the headers alone.

``inspect(frame)`` -> dict with ``fcs_bytes`` (size of the Frame_Content_Size field, 1 for the single-segment
one-byte form), ``blocks`` (one dict per block: ``type`` raw / rle / compressed; for compressed blocks
``literals`` raw / rle / huffman / treeless, ``streams`` 1 or 4, ``modes`` of the LL, OF and ML tables among
predefined / rle / fse / repeat (None when the block has no sequences) and ``modes_at``, where that modes byte
is, and ``huf_streams``, the byte range of the frame its Huffman streams occupy).  Any frame libzstd writes
parses; no entropy data is decoded."""

LIT_TYPES = ('raw', 'rle', 'huffman', 'treeless')
MODES = ('predefined', 'rle', 'fse', 'repeat')
BLOCK_TYPES = ('raw', 'rle', 'compressed', 'reserved')


def _literals(b, p):
    """(info, size of the literals section) of the compressed block starting at b[p]."""
    t, lh = b[p] & 3, (b[p] >> 2) & 3
    if t < 2:
        hs = {0: 1, 2: 1, 1: 2, 3: 3}[lh]
        size = int.from_bytes(b[p:p + hs], 'little') >> (3 if hs == 1 else 4)
        return dict(literals=LIT_TYPES[t], streams=1, huf_streams=None), hs + (size if t == 0 else 1)
    hs = {0: 3, 1: 3, 2: 4, 3: 5}[lh]
    v = int.from_bytes(b[p:p + hs], 'little')
    csize = v >> {3: 14, 4: 18, 5: 22}[hs]
    tree = 0
    if t == 2:
        w = b[p + hs]
        tree = 1 + (w if w < 128 else (w - 127 + 1) // 2)
    return (dict(literals=LIT_TYPES[t], streams=1 if lh == 0 else 4, huf_streams=(p + hs + tree, p + hs + csize)),
            hs + csize)


def inspect(frame: bytes) -> dict:
    b = frame
    assert int.from_bytes(b[:4], 'little') == 0xFD2FB528, 'not a zstd frame'
    fhd = b[4]
    single, fcs_id, did = (fhd >> 5) & 1, fhd >> 6, fhd & 3
    fcs_bytes = (0, 2, 4, 8)[fcs_id] or (1 if single else 0)
    p = 5 + (not single) + (0, 1, 2, 4)[did] + fcs_bytes
    blocks = []
    while True:
        h = int.from_bytes(b[p:p + 3], 'little')
        p += 3
        last, btype, size = h & 1, BLOCK_TYPES[(h >> 1) & 3], h >> 3
        blk = dict(type=btype, start=p)
        if btype == 'compressed':
            lit, n = _literals(b, p)
            blk.update(lit)
            q = p + n
            nseq = b[q]
            q += 1 if nseq < 128 else 2 if nseq < 255 else 3
            blk['modes'] = blk['modes_at'] = None
            if nseq:
                m = b[q]
                blk['modes_at'] = q
                blk['modes'] = dict(LL=MODES[m >> 6], OF=MODES[(m >> 4) & 3], ML=MODES[(m >> 2) & 3])
        blocks.append(blk)
        p += 1 if btype == 'rle' else size
        if last:
            break
    return dict(fcs_bytes=fcs_bytes, checksum=bool(fhd & 4), blocks=blocks, end=p)
