"""Per-read caller: the reference's ``WarpSTR`` seam on top of the batched GPU engine.

Mirrors caller/caller.py of the reference: ``CallerResult`` (:46-51), ``WarpResult``
(:54-63), ``WarpSTR(flank_length, states, endstate, repeat_mask, out_warp_path, reverse,
read_name).run(signal) / .warp(signal, mask)`` (:107-193).  The DP fill and traceback of
both passes run in the CUDA kernels behind ``wstr_warp_batch``; :class:`CallerEngine`
batches reads so that thousands of them are in flight at once.
"""
import hashlib
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence

import numpy as np

from . import _lib, midstage
from .config import CallerConfig, RescalerConfig
from .templates import reverse_complement


@dataclass
class CallerResult:
    seq: str
    cost: float
    resc_seq: str
    resc_cost: float


@dataclass
class WarpResult:
    trace: np.ndarray

    @property
    def state_transitions(self) -> np.ndarray:
        keep = np.concatenate(([True], self.trace[1:] != self.trace[:-1]))
        return self.trace[keep]


@dataclass
class NotLocated:
    """In place of a CallerResult: the read's STR window was not found in the whole read (DESIGN.md section
    4.5), so the read was not called.  ``status`` is _lib.LOCATE_NOT_FOUND (the best window scores >= 0) or
    _lib.LOCATE_NO_PATH (the read is shorter than the automaton's shortest path)."""
    status: int
    score: float


def choose_strand(status, score):
    """The strand of reads searched on both strands (DESIGN.md section 4.5).  ``status`` / ``score``: (n, 2), column
    0 the template automaton's search, column 1 the reverse automaton's.  The rule:

    * found (_lib.LOCATE_FOUND) on one strand only: that strand;
    * found on both: the lower score; an exact tie goes to the template (no margin);
    * found on neither: no strand (-1), status LOCATE_NOT_FOUND if either search had it, else LOCATE_NO_PATH,
      and the lower score.

    Returns (strand int8[n]: 0 template, 1 reverse, -1 neither; col int64[n]: the column the window and score
    come from, the lower score's (template on a tie) where neither is found; status int32[n]; score float64[n])."""
    status = np.asarray(status).reshape(-1, 2)
    score = np.asarray(score, dtype=np.float64).reshape(-1, 2)
    found = status == _lib.LOCATE_FOUND
    lower_rev = score[:, 1] < score[:, 0]
    both, neither = found.all(axis=1), ~found.any(axis=1)
    col = np.where(both | neither, lower_rev, found[:, 1]).astype(np.int64)
    strand = np.where(neither, -1, col).astype(np.int8)
    st = np.where(neither, np.where((status == _lib.LOCATE_NOT_FOUND).any(axis=1), _lib.LOCATE_NOT_FOUND,
                                    _lib.LOCATE_NO_PATH), _lib.LOCATE_FOUND).astype(np.int32)
    return strand, col, st, score[np.arange(len(col)), col]


HIT_FIELDS = ('read', 'locus', 'strand', 'left_lo', 'left_hi', 'left_score', 'right_lo', 'right_hi', 'right_score')


def hit_arrays(hits) -> Dict[str, np.ndarray]:
    """wstr_assign_hit records (_lib.ASSIGN_HIT, any order) -> one array per field of HIT_FIELDS, sorted by
    (read, locus)."""
    order = np.lexsort((hits['locus'], hits['read']))
    return {f: np.ascontiguousarray(hits[f][order]) for f in HIT_FIELDS}


def split_pairs(aut):
    """Per read one automaton id or a (template id, reverse id) pair -> (pair bool[n], ids int32[n, 2]); a read
    given one id has it in both columns."""
    if isinstance(aut, np.ndarray) and aut.ndim == 1:
        ids = aut.astype(np.int32)
        return np.zeros(len(ids), dtype=bool), np.stack((ids, ids), axis=1)
    n = len(aut)
    ids = np.empty((n, 2), dtype=np.int32)
    pair = np.zeros(n, dtype=bool)
    for r, a in enumerate(aut):
        if np.ndim(a) == 0:
            ids[r] = int(a)
        else:
            ids[r] = [int(x) for x in a]
            pair[r] = True
    return pair, ids


def fill_given_strands(loc, reverse) -> None:
    """Completes ``loc['strand']`` of a locate dict: a read with a given strand (``reverse[r]`` a bool; None for a
    read searched on both strands) gets that strand, found or not."""
    given = np.array([r is not None for r in reverse], dtype=bool)
    rv = np.array([bool(r) if r is not None else False for r in reverse], dtype=np.int8)
    loc['strand'] = np.where(given, rv, loc['strand']).astype(np.int8)


_SCALARS = ('len1', 'len2', 'cost1', 'cost2', 'status', 'ties')      # per-read results of a call

# exception types the reference raises for a read, by d_status code
_STATUS_ERRORS = {
    1: (IndexError, 'index out of bounds: signal shorter than min_values_per_state + 1'),
    2: (RuntimeError, 'Unexpected error during backtracking'),
}


def pack_signals(signals: Sequence[np.ndarray]):
    """Concatenate reads into one float64 buffer with 16-byte aligned starts.
    Returns (pinned host tensor, offsets int64[n], lengths int32[n])."""
    import torch
    n = len(signals)
    lengths = np.fromiter((len(s) for s in signals), dtype=np.int32, count=n)
    offsets, total = even_offsets(lengths)
    host = torch.empty(total, dtype=torch.float64, pin_memory=torch.cuda.is_available())
    buf = host.numpy()
    for s, o, ln in zip(signals, offsets, lengths):
        buf[o:o + ln] = s
        if ln & 1:
            buf[o + ln] = 0.0
    buf[total - 2:] = 0.0
    return host, offsets, lengths


def pack_masks(masks: Sequence[np.ndarray]):
    """Bit-pack per-read bool masks, 32 rows per little-endian word.
    Returns (host uint32 array, word offsets int64[n])."""
    n = len(masks)
    nwords = np.fromiter(((len(m) + 31) // 32 for m in masks), dtype=np.int64, count=n)
    offsets = np.zeros(n, dtype=np.int64)
    if n > 1:
        offsets[1:] = np.cumsum(nwords[:-1])
    out = np.zeros(int(nwords.sum()) + 1, dtype=np.uint32)
    for m, o, w in zip(masks, offsets, nwords):
        bits = np.packbits(np.asarray(m, dtype=bool), bitorder='little')
        pad = (-len(bits)) % 4
        if pad:
            bits = np.concatenate((bits, np.zeros(pad, dtype=np.uint8)))
        out[o:o + w] = bits.view('<u4')
    return out, offsets


def even_offsets(lengths: np.ndarray):
    """Element offsets of float64 windows packed with 16-byte aligned starts, and the buffer size."""
    padded = (lengths.astype(np.int64) + 1) & ~1
    off = np.zeros(len(lengths), dtype=np.int64)
    if len(lengths) > 1:
        off[1:] = np.cumsum(padded[:-1])
    return off, int(padded.sum()) + 2


def _span(off, lengths, a, b, size):
    """Element range [lo, hi) of reads [a, b) (b > a) in a float64 buffer of ``size`` elements packed as
    ``even_offsets`` packs them: up to 2 elements past the last read's even end (the kernels read that far),
    clipped at the buffer's end."""
    return int(off[a]), min(int(off[b - 1] + ((int(lengths[b - 1]) + 1) & ~1) + 2), size)


def _window_bounds(raw_off, win_lo, win_hi):
    """(lo int32[n], hi int32[n], lengths int32[n]) of the windows ``[win_lo, win_hi]`` (inclusive) of whole
    reads at offsets ``raw_off`` (int64[n + 1]): a window is clipped at its read's end like a numpy slice; a
    negative start raises ValueError."""
    lo = np.asarray(win_lo, dtype=np.int32)
    hi = np.asarray(win_hi, dtype=np.int32)
    if (lo < 0).any():
        raise ValueError('negative window start')
    lengths = np.maximum(np.minimum(hi.astype(np.int64), np.diff(raw_off) - 1) - lo + 1, 0).astype(np.int32)
    return lo, hi, lengths


def _nothing(self, *args):
    """The hook of an ingest form or whole-read source that has nothing to do at that step."""


class _IngestF64:
    """Host float64 windows (the reference's ReadSignal.signal): copied as they are."""

    def __init__(self, eng, host_signal, off, lengths):
        self.eng, self.host, self.sig_off, self.lengths = eng, host_signal, off, lengths
        self.total = _span(off, lengths, 0, len(lengths), host_signal.numel())[1] if len(lengths) else 0
        self.h2d_bytes = self.total * 8

    def allocate(self):
        import torch
        self.d_sig = self.eng._device_buffer('sig', self.total, torch.float64)

    def send(self, a, b):
        lo, hi = _span(self.sig_off, self.lengths, a, b, self.d_sig.numel())
        self.d_sig[lo:hi].copy_(self.host[lo:hi], non_blocking=True)

    prepare = fetch = finish = _nothing


class _IngestI16:
    """Host int16 window samples + {shift, scale} per read; float64 windows are made on the device."""

    def __init__(self, eng, host_raw, raw_off, lengths, host_ss):
        self.eng, self.host, self.raw_off, self.lengths, self.host_ss = eng, host_raw, raw_off, lengths, host_ss
        self.sig_off, self.total = even_offsets(lengths)
        self.h2d_bytes = int(host_raw.numel()) * 2 + int(host_ss.numel()) * 8

    def allocate(self):
        import torch
        e = self.eng
        self.d_sig = e._device_buffer('sig', self.total, torch.float64)
        self.d_raw = e._device_buffer('raw16', int(self.host.numel()), torch.int16)
        self.d_ss = e._device_buffer('shift_scale', 2 * len(self.lengths), torch.float64)

    def _raw_range(self, a, b):
        return int(self.raw_off[a]), min(int(self.raw_off[b - 1] + self.lengths[b - 1]), int(self.host.numel()))

    def send(self, a, b):
        lo, hi = self._raw_range(a, b)
        self.d_raw[lo:hi].copy_(self.host[lo:hi], non_blocking=True)
        self.d_ss[2 * a:2 * b].copy_(self.host_ss.reshape(-1)[2 * a:2 * b], non_blocking=True)

    def prepare(self, a, b, lane):
        import torch
        ws = self.eng._device_buffer(f'deq_ws{lane}', 24 * (b - a) + 256, torch.uint8)
        _lib.dequantize_batch(self.d_raw, self.raw_off[a:b], self.lengths[a:b], self.d_ss[2 * a:2 * b], self.d_sig,
                              self.sig_off[a:b], ws)

    fetch = finish = _nothing


def pack_raw(raws):
    """Whole int16 reads -> one pinned host buffer and the read offsets (int64[n + 1])."""
    import torch
    n = len(raws)
    lens = np.fromiter((len(r) for r in raws), dtype=np.int64, count=n)
    if (lens <= 0).any():
        raise ValueError('empty raw read')
    raw_off = np.zeros(n + 1, dtype=np.int64)
    raw_off[1:] = np.cumsum(lens)
    host = torch.empty(int(raw_off[-1]), dtype=torch.int16, pin_memory=torch.cuda.is_available())
    hb = host.numpy()
    for r, o in zip(raws, raw_off[:-1]):
        hb[o:o + len(r)] = np.asarray(r, dtype=np.int16)
    return host, raw_off


def pack_vbz(reads):
    """Chunks of compressed reads (fast5.CompressedRead) -> what ``call_arrays_vbz`` takes: the pinned payload
    buffer (every chunk's payload at a 16-byte aligned offset, zero padded: the decoders read whole 16-byte
    words), the chunk table, the first chunk of every read (int64[n + 1]) and the read offsets in the
    decoded int16 buffer (int64[n + 1]).

    A chunk that is still a zstd frame (fast5.KIND_VBZ*_ZSTD) is uploaded as the frame: its table row has
    ``zstd_off`` / ``zstd_bytes``, the frame's place in the payload, and ``in_off`` / ``in_bytes`` name where
    wstr_zstd_decode_batch writes its body, in a region of the device buffer behind the uploaded bytes (the
    decoded-body region, ``device_bytes`` in all).  Other rows have ``zstd_off`` -1 and are read where they
    were uploaded, so every StreamVByte body is read from the one device buffer."""
    import torch
    from .fast5 import KIND_RAW, KIND_VBZ0_ZSTD
    chunks = [c for r in reads for c in r.chunks]
    m = len(chunks)
    n_chunks = np.fromiter((len(r.chunks) for r in reads), dtype=np.int64, count=len(reads))
    read_chunk = np.zeros(len(reads) + 1, dtype=np.int64)
    read_chunk[1:] = np.cumsum(n_chunks)
    raw_off = np.zeros(len(reads) + 1, dtype=np.int64)
    raw_off[1:] = np.cumsum(np.fromiter((r.n_samples for r in reads), dtype=np.int64, count=len(reads)))
    kind = np.fromiter((c.kind for c in chunks), dtype=np.int32, count=m)
    frame = kind >= KIND_VBZ0_ZSTD
    up_bytes = np.fromiter((len(c.payload) for c in chunks), dtype=np.int64, count=m)
    up_off = np.zeros(m + 1, dtype=np.int64)
    up_off[1:] = np.cumsum((up_bytes + 15) & ~15)
    body = np.where(frame, np.fromiter((c.body_size for c in chunks), dtype=np.int64, count=m), 0)
    body_off = np.zeros(m + 1, dtype=np.int64)
    body_off[1:] = np.cumsum((body + 15) & ~15)
    chunk_read = np.repeat(np.arange(len(reads)), n_chunks)
    table = dict(in_off=np.where(frame, int(up_off[-1]) + body_off[:-1], up_off[:-1]),
                 in_bytes=np.where(frame, body, up_bytes),
                 n_samples=np.fromiter((c.coded if c.kind != KIND_RAW else c.count for c in chunks), dtype=np.int32,
                                       count=m),
                 n_out=np.fromiter((c.count for c in chunks), dtype=np.int32, count=m),
                 kind=np.where(frame, kind - KIND_VBZ0_ZSTD, kind).astype(np.int32),
                 zigzag=np.fromiter((c.zigzag for c in chunks), dtype=np.int32, count=m),
                 out_off=raw_off[chunk_read] + np.fromiter((c.start for c in chunks), dtype=np.int64, count=m),
                 zstd_off=np.where(frame, up_off[:-1], -1), zstd_bytes=np.where(frame, up_bytes, 0))
    host = torch.zeros(max(int(up_off[-1]), 16), dtype=torch.uint8, pin_memory=torch.cuda.is_available())
    hb = host.numpy()
    for c, o in zip(chunks, up_off[:-1]):
        hb[o:o + len(c.payload)] = np.frombuffer(c.payload, dtype=np.uint8)
    return host, table, read_chunk, raw_off


class _WholeReads:
    """Whole int16 reads in a pinned host buffer as ``pack_raw`` lays them out, or already on the device (``d_raw``,
    nothing to send).  ``samples(idx)``: the host samples of reads ``idx``, for the host redo.  ``_VBZReads`` is the
    other form; both allocate, send and decode reads [a, b) on the current stream, fetch the decode statuses, put
    them into a result (``finish``) and raise the first bad chunk's error from it (``raise_bad``)."""

    def __init__(self, host, raw_off, d_raw=None, samples=None):
        self.host, self.d_raw, self.samples = host, d_raw, samples
        self.raw_off = np.asarray(raw_off, dtype=np.int64)
        self.h2d_bytes = int(self.raw_off[-1]) * 2 if host is not None else 0

    def allocate(self, eng, name):
        import torch
        if self.host is not None:
            self.d_raw = eng._device_buffer(name, int(self.raw_off[-1]), torch.int16)

    def send(self, a, b):
        if self.host is not None:
            lo, hi = int(self.raw_off[a]), int(self.raw_off[b])
            self.d_raw[lo:hi].copy_(self.host[lo:hi], non_blocking=True)

    decode = fetch = finish = raise_bad = _nothing     # int16 reads need no decode and have no statuses


class _VBZReads(_WholeReads):
    """Whole reads as VBZ chunks, as ``pack_vbz`` lays them out: the payload crosses the host link as stored,
    zstd frames are decoded on the device (wstr_zstd_decode_batch), then the StreamVByte / delta decode
    (wstr_vbz_decode_batch) writes the int16 reads.  The statuses: WSTR_VBZ_* per chunk and WSTR_ZSTD_* per
    frame, frames numbered in chunk order, in one pinned buffer laid out [chunks | frames]."""

    def __init__(self, host_payload, table, read_chunk, raw_off, reads=None):
        super().__init__(None, raw_off, samples=lambda idx: [reads[r].decode() for r in idx])
        self.payload, self.table, self.reads = host_payload, table, reads
        self.read_chunk = np.asarray(read_chunk, dtype=np.int64)
        frame = np.asarray(table['zstd_off']) >= 0
        self.frame_rows = np.flatnonzero(frame)                  # table rows of the zstd frames
        self.frame_of = np.zeros(len(frame) + 1, dtype=np.int64)  # frames before chunk c
        self.frame_of[1:] = np.cumsum(frame)
        # the chunks are uploaded one after the other at 16-byte aligned offsets: a frame at zstd_off (its body is
        # decoded to in_off, behind the uploaded bytes), any other chunk at in_off
        in_end = table['in_off'] + ((table['in_bytes'] + 15) & ~15)
        up_end = np.where(frame, table['zstd_off'] + ((table['zstd_bytes'] + 15) & ~15), in_end)
        self.pay_off = np.append(0, up_end)[self.read_chunk]   # uploaded bytes of reads [a, b)
        self.h2d_bytes = int(self.pay_off[-1])
        self.device_bytes = max(int(host_payload.numel()), int(in_end.max()) if len(in_end) else 0, 16)

    def allocate(self, eng, name):
        import torch
        m, nf = len(self.frame_of) - 1, len(self.frame_rows)
        self.d_raw = eng._device_buffer(name, int(self.raw_off[-1]), torch.int16)
        self.d_payload = eng._device_buffer('vbz_payload', self.device_bytes, torch.uint8)
        self.d_status = eng._device_buffer('vbz_status', m, torch.int32)
        self.d_zstatus = eng._device_buffer('zstd_status', max(nf, 1), torch.int32)
        self.h_status = eng._host_buffer('vbz_status', m + nf, torch.int32)

    def send(self, a, b):
        lo, hi = int(self.pay_off[a]), int(self.pay_off[b])
        self.d_payload[lo:hi].copy_(self.payload[lo:hi], non_blocking=True)

    def _ranges(self, a, b):
        """Chunks [c0, c1) and frames [f0, f1) of reads [a, b)."""
        c0, c1 = int(self.read_chunk[a]), int(self.read_chunk[b])
        return c0, c1, int(self.frame_of[c0]), int(self.frame_of[c1])

    def decode(self, eng, a, b, lane):
        import torch
        c0, c1, f0, f1 = self._ranges(a, b)
        if f1 > f0:
            rows, t = self.frame_rows[f0:f1], self.table
            ws = eng._device_buffer(f'zstd_ws{lane}', _lib.zstd_workspace_bytes(f1 - f0), torch.uint8)
            _lib.zstd_decode_batch(self.d_payload, t['zstd_off'][rows], t['zstd_bytes'][rows], t['in_off'][rows],
                                   t['in_bytes'][rows], self.d_payload, self.d_zstatus[f0:f1], ws)
        if c1 > c0:
            t = {k: v[c0:c1] for k, v in self.table.items()}
            ws = eng._device_buffer(f'vbz_ws{lane}', _lib.vbz_workspace_bytes(c1 - c0), torch.uint8)
            _lib.vbz_decode_batch(self.d_payload, t['in_off'], t['in_bytes'], t['n_samples'], t['n_out'], t['kind'],
                                  t['zigzag'], t['out_off'], self.d_raw, self.d_status[c0:c1], ws)

    def fetch(self, a, b):
        c0, c1, f0, f1 = self._ranges(a, b)
        m = len(self.frame_of) - 1
        self.h_status[c0:c1].copy_(self.d_status[c0:c1], non_blocking=True)
        if f1 > f0:
            self.h_status[m + f0:m + f1].copy_(self.d_zstatus[f0:f1], non_blocking=True)

    def finish(self, res):
        """``chunk_status`` and ``zstd_status`` (per chunk, 0 for a chunk that was not a zstd frame) into ``res``;
        the fetches must have completed."""
        m = len(self.frame_of) - 1
        h = self.h_status.numpy()
        res['chunk_status'], res['zstd_status'] = h[:m].copy(), np.zeros(m, dtype=np.int32)
        res['zstd_status'][self.frame_rows] = h[m:]

    def raise_bad(self, res):
        """Takes the statuses out of ``res`` and raises the Fast5FormatError of the first chunk the device decoders
        refused, naming the file and the read: a zstd frame they refuse raises the host decoder's own 'zstd:
        corrupt VBZ chunk'."""
        from .fast5 import Fast5FormatError
        chunk_status, zst = res.pop('chunk_status'), res.pop('zstd_status')
        bad = np.flatnonzero((chunk_status != 0) | (zst != 0))
        if len(bad):
            c = int(bad[0])
            r = int(np.searchsorted(self.read_chunk, c, side='right')) - 1
            read = self.reads[r]
            msg = ('zstd: corrupt VBZ chunk' if zst[c] else
                   _lib.VBZ_STATUS_MESSAGES.get(int(chunk_status[c]), 'VBZ: corrupt chunk'))
            raise Fast5FormatError(f'{read.path}: read {read.read_name}: {msg} '
                                   f'(chunk at sample {read.chunks[c - int(self.read_chunk[r])].start})')


class _IngestRaw:
    """Whole int16 reads (a ``_WholeReads``) + windows: the source's decode, then spike removal, MAD
    normalisation and slicing on the device."""

    def __init__(self, eng, src, lo, hi, lengths, spike_mode):
        self.eng, self.src, self.lo, self.hi = eng, src, lo, hi
        self.lengths, self.spike_mode = lengths, spike_mode
        self.sig_off, self.total = even_offsets(lengths)
        self.h2d_bytes, self.send = src.h2d_bytes, src.send

    def allocate(self):
        import torch
        e, n = self.eng, len(self.lengths)
        self.d_sig = e._device_buffer('sig', self.total, torch.float64)
        self.src.allocate(e, 'raw16')
        self.d_ss = e._device_buffer('shift_scale', 2 * n, torch.float64)
        self.h_ss = e._host_buffer('shift_scale', 2 * n, torch.float64)

    def prepare(self, a, b, lane):
        import torch
        self.src.decode(self.eng, a, b, lane)
        ws = self.eng._device_buffer(f'norm_ws{lane}', _lib.normalize_workspace_bytes(b - a), torch.uint8)
        _lib.normalize_batch(self.src.d_raw, self.src.raw_off[a:b + 1], self.lo[a:b], self.hi[a:b], self.spike_mode,
                             self.d_sig, self.sig_off[a:b], self.d_ss[2 * a:2 * b], ws)

    def fetch(self, a, b):
        self.h_ss[2 * a:2 * b].copy_(self.d_ss[2 * a:2 * b], non_blocking=True)
        self.src.fetch(a, b)

    def finish(self, res):
        res['shift_scale'] = self.h_ss.numpy().reshape(-1, 2).copy()
        res['lengths'] = self.lengths
        self.src.finish(res)


class CallerEngine:
    """Batched two-pass WarpSTR caller on one GPU."""

    def __init__(self, caller_config: Optional[CallerConfig] = None,
                 rescaler_config: Optional[RescalerConfig] = None, device: str = 'cuda',
                 workspace_bytes: Optional[int] = None):
        import torch
        if not torch.cuda.is_available():
            raise _lib.WarpstrError('warpstr_b200 needs a CUDA device (there is no CPU fallback)')
        _lib.lib()
        self.cc = caller_config or CallerConfig()
        self.rc = rescaler_config or RescalerConfig()
        self.device = torch.device(device)
        self.workspace_limit = workspace_bytes
        self.automata: List[_lib.DeviceAutomaton] = []
        self.tables: List[dict] = []
        self._lane_ws = {}
        self._streams = {}
        self.timeline = None      # set to a list to collect (label, CUDA event) pairs from call_arrays
        self._dev_cache = {}
        self._host_cache = {}
        self._h2d_probe = None
        self.split_small = (4096, 40000)   # batch sizes a resident call runs as two concurrent halves (None: never)
        self.ttest_guard_ulps = 0    # 0 = the library's default (16 ulp), see wstr_call_outputs.d_ttest_ties
        self.last_ttest_ties = 0     # reads of the last results_from() that were re-evaluated for a t-test tie
        self.last_located = None     # windows of the last call_*_batch(windows=None): dict as from locate_packed

    # -- automata ------------------------------------------------------------------------
    def add_automaton(self, sta, flank_length: int) -> int:
        """Upload one strand's automaton (object with values/seq_idx/in_ptr/in_idx/rep_mask/
        last_base/endstate, e.g. warpstr_b200.automata.StateAutomata); returns its id."""
        import torch
        with torch.cuda.device(self.device):
            dev = _lib.DeviceAutomaton.from_automaton(sta, flank_length, self.cc.min_values_per_state)
        self.automata.append(dev)
        self.tables.append(dict(values=np.asarray(sta.values, dtype=np.float64),
                                seq_idx=np.asarray(sta.seq_idx), rep_mask=np.asarray(sta.rep_mask, dtype=bool),
                                last_base=bytes(np.asarray(sta.last_base, dtype=np.uint8)).decode('ascii'),
                                flank_length=int(flank_length)))
        return len(self.automata) - 1

    # -- device helpers ---------------------------------------------------------------------
    def _workspace(self, need: int, lane: int = 0):
        """Device workspace of ``need`` bytes for compute lane ``lane`` (each lane of the pipelined call owns
        one, sized for its chunks), or as much as the memory limit allows (the library then works in waves):
        the explicit limit, else 60 % of what is free.  The buffer only grows; cudaMemGetInfo is asked only
        when it has to (the call can block for tens of milliseconds while the GPU is busy)."""
        import torch
        ws, at_limit, need_seen = self._lane_ws.get(lane, (None, False, 0))
        if ws is not None and (ws.numel() >= need or (at_limit and need <= need_seen)):
            return ws
        limit = self.workspace_limit
        if limit is None:
            free, _ = torch.cuda.mem_get_info(self.device)
            limit = int(free * 0.6) + (ws.numel() if ws is not None else 0)
        size = min(need, max(limit, 1 << 20))
        if ws is None or ws.numel() < size:
            ws = torch.empty(size, dtype=torch.uint8, device=self.device)
        # a larger request re-evaluates the limit (memory may have been freed)
        self._lane_ws[lane] = (ws, size < need, need)
        return ws

    def warp_batch(self, signals: Sequence[np.ndarray], aut_ids: Sequence[int],
                   masks: Optional[Sequence[np.ndarray]] = None, return_end_cost: bool = False):
        """One DP pass + traceback for every read (reference: WarpSTR.warp, caller.py:189-193).
        Returns the list of traces (int32 state index per sample)."""
        import torch
        n = len(signals)
        if n == 0:
            return ([], np.zeros(0)) if return_end_cost else []
        with torch.cuda.device(self.device):
            host, off, lengths = pack_signals(signals)
            d_sig = host.to(self.device, non_blocking=True)
            aut = np.asarray(aut_ids, dtype=np.int32)
            d_mask, moff = None, None
            if masks is not None:
                hm, moff = pack_masks(masks)
                d_mask = torch.from_numpy(hm.view(np.int32)).to(self.device)
            need = _lib.warp_workspace_bytes(self.automata, aut, lengths)
            ws = self._workspace(need)
            d_trace = torch.empty(d_sig.numel(), dtype=torch.int32, device=self.device)
            d_status = torch.zeros(n, dtype=torch.int32, device=self.device)
            d_cost = torch.empty(n, dtype=torch.float64, device=self.device) if return_end_cost else None
            _lib.warp_batch(self.automata, aut, d_sig, off, lengths, d_mask, moff, ws, d_trace, d_cost, d_status)
            trace = d_trace.cpu().numpy()
            status = d_status.cpu().numpy()
        for r in np.flatnonzero(status):
            exc, msg = _STATUS_ERRORS.get(int(status[r]), (RuntimeError, f'read failed with status {status[r]}'))
            raise exc(msg)
        traces = [trace[o:o + ln] for o, ln in zip(off, lengths)]
        if return_end_cost:
            return traces, d_cost.cpu().numpy()
        return traces

    # -- full two-pass call ----------------------------------------------------------------
    def decode(self, aut_id: int, runs: midstage.Runs, reverse: bool) -> str:
        """caller.py:178-187: last base of each run's k-mer, flanks trimmed."""
        tb = self.tables[aut_id]
        seq = ''.join(tb['last_base'][s] for s in runs.states)
        offset = int(tb['seq_idx'][runs.states[0]])
        F = tb['flank_length']
        seq = seq[F - offset:-F]
        return reverse_complement(seq) if reverse else seq

    def call_batch(self, signals: Sequence[np.ndarray], aut_ids: Sequence[int],
                   reverse: Sequence[bool], engine: Optional[str] = None) -> List[CallerResult]:
        """WarpSTR.run for a batch (caller.py:117-149).  ``engine='gpu'`` (the default) keeps everything
        on the device (wstr_call_batch); ``engine='host'`` runs the two DP passes on the GPU and the
        stage between them with numpy/scipy on the host -- the evaluation used for reads the device
        flags (a t-test tie, a spline that needs interior knots, a reference exception)."""
        signals = [np.ascontiguousarray(s, dtype=np.float64) for s in signals]
        engine = engine or 'gpu'
        if engine == 'host':
            return self._call_batch_host(signals, aut_ids, reverse)
        res = self.call_packed(*self.upload(signals, aut_ids, reverse))
        return self.results_from(res, signals, aut_ids, reverse)

    # -- device-resident form -----------------------------------------------------------------------
    def upload(self, signals: Sequence[np.ndarray], aut_ids: Sequence[int], reverse: Sequence[bool]):
        """Host -> device copy of a batch.  Returns the tuple ``call_packed`` takes."""
        host, off, lengths = pack_signals(signals)
        d_sig = host.to(self.device, non_blocking=True)
        return d_sig, off, lengths, np.asarray(aut_ids, dtype=np.int32), np.asarray(reverse, dtype=np.uint8)

    def call_packed(self, d_sig, off, lengths, aut, rev, want_seq: bool = True, want_debug: bool = False,
                    into: Optional[dict] = None, lane: int = 0, allow_split: bool = True):
        """wstr_call_batch on device-resident signals.  Returns a dict of device tensors
        (len1, len2, cost1, cost2, status, ties[, seq1, seq2, seq_off]).  A batch whose per-batch buffers
        (rescaled signal, traces, mid-stage scratch: ~35 B per sample) do not fit the workspace the memory
        allows is cut into consecutive slices, one library call each."""
        import torch
        n = len(lengths)
        lengths = np.asarray(lengths, dtype=np.int32)
        off = np.asarray(off, dtype=np.int64)
        aut = np.asarray(aut, dtype=np.int32)
        rev = np.asarray(rev, dtype=np.uint8)
        with torch.cuda.device(self.device):
            need = _lib.call_workspace_bytes(self.automata, aut, lengths)
            ws = self._workspace(need, lane)
            if into is not None:      # caller-owned result buffers (views of the right sizes)
                o = dict(into)
                o['status'].zero_()
                if 'ties' in o:
                    o['ties'].zero_()
            else:
                o = dict(
                    len1=torch.empty(n, dtype=torch.int32, device=self.device),
                    len2=torch.empty(n, dtype=torch.int32, device=self.device),
                    cost1=torch.empty(n, dtype=torch.float64, device=self.device),
                    cost2=torch.empty(n, dtype=torch.float64, device=self.device),
                    status=torch.zeros(n, dtype=torch.int32, device=self.device),
                    ties=torch.zeros(n, dtype=torch.int32, device=self.device))
            seq_off = None
            if want_seq:
                cap = lengths.astype(np.int64) // max(self.cc.min_values_per_state - 1, 1) + 16
                seq_off = np.zeros(n, dtype=np.int64)
                seq_off[1:] = np.cumsum(cap[:-1])
                total = int(cap.sum())
                if into is None:
                    # zeroed for the parity tests (want_debug), as the buffers below: a read's sequence fills only
                    # part of its capacity, the rest is never written, and the tests compare whole buffers
                    alloc = torch.zeros if want_debug else torch.empty
                    o['seq1'] = alloc(total, dtype=torch.uint8, device=self.device)
                    o['seq2'] = alloc(total, dtype=torch.uint8, device=self.device)
                o['seq_off'] = seq_off
            if want_debug:   # intermediate products, for the parity tests
                # (zeroed: the padding between reads is never written, and the tests compare whole buffers; left
                # uninitialised it holds whatever an earlier call freed)
                o['trace1'] = torch.zeros(d_sig.numel(), dtype=torch.int32, device=self.device)
                o['trace2'] = torch.zeros(d_sig.numel(), dtype=torch.int32, device=self.device)
                o['rescaled'] = torch.zeros(d_sig.numel(), dtype=torch.float64, device=self.device)
            params = _lib.CallParams(self.cc.min_values_per_state, self.cc.states_in_segment,
                                     float(self.rc.threshold), float(self.rc.max_std),
                                     1 if self.rc.method == 'median' else 0, 1 if self.rc.reps_as_one else 0,
                                     int(self.ttest_guard_ulps))
            def run(a, b, wsp, stream):
                lo, hi = _span(off, lengths, a, b, d_sig.numel())
                sl = slice(lo, hi)

                def part(key, x0, x1):
                    t = o.get(key)
                    return t[x0:x1] if t is not None else None
                s0 = int(seq_off[a]) if want_seq else 0
                _lib.call_batch(self.automata, aut[a:b], rev[a:b], d_sig[sl], off[a:b] - lo, lengths[a:b], params, wsp,
                                o['len1'][a:b], o['len2'][a:b], o['cost1'][a:b], o['cost2'][a:b], o['status'][a:b],
                                part('seq1', s0, None), part('seq2', s0, None),
                                seq_off[a:b] - s0 if want_seq else None,
                                part('trace1', lo, hi), part('trace2', lo, hi), part('rescaled', lo, hi),
                                stream=stream, d_ttest_ties=o['ties'][a:b] if 'ties' in o else None)

            halves = self._halves(n, lane) if allow_split else None
            if halves is not None:
                # A small batch is a handful of rounds of the resident warps, the last one partly empty, and
                # four launches in a row each with such a tail.  Two halves on two streams fill each other's
                # gaps: one half's mid-stage and kernel tails run under the other half's DP.
                mid, side = halves
                cur = torch.cuda.current_stream()
                need2 = _lib.call_workspace_bytes(self.automata, aut[mid:], lengths[mid:])
                ws2 = self._workspace(need2, 1)
                side.wait_stream(cur)
                run(0, mid, ws, None)
                run(mid, n, ws2, side)
                cur.wait_stream(side)
            else:
                for a, b in self._slices(ws.numel(), need, aut, lengths):
                    run(a, b, ws, None)
        return o

    def _halves(self, n: int, lane: int):
        """(split point, side stream) when a resident call should run as two concurrent halves."""
        if lane != 0 or not self.split_small or not (self.split_small[0] <= n <= self.split_small[1]):
            return None
        return n // 2, self._side_streams('lanes')[0]

    def _side_streams(self, group: str):
        """The engine's side streams: 'lanes', three compute lanes beside the current stream, or 'copy', the
        pipeline's input and result streams.  Each group is taken from torch's stream pool when a call first needs
        it (the pool index decides which hardware queue a stream shares)."""
        import torch
        if group not in self._streams:
            self._streams[group] = [torch.cuda.Stream() for _ in range(3 if group == 'lanes' else 2)]
        return self._streams[group]

    def _slices(self, ws_bytes: int, need: int, aut, lengths):
        """Consecutive read ranges of one call_packed: the whole batch when the workspace holds what a call
        needs per batch (the direction codes may still go in waves), else slices that leave half of the
        workspace to the direction codes."""
        n = len(lengths)
        if n == 0:
            return []
        if need <= ws_bytes or _lib.call_workspace_min_bytes(self.automata, aut, lengths) <= ws_bytes // 2:
            return [(0, n)]
        parts = 2
        while True:
            cum = np.cumsum(lengths.astype(np.int64))
            cuts = np.searchsorted(cum, cum[-1] * np.arange(1, parts) / parts, side='right')
            bounds = sorted(set([0] + [int(c) for c in cuts] + [n]))
            pairs = [(a, b) for a, b in zip(bounds[:-1], bounds[1:]) if b > a]
            if all(_lib.call_workspace_min_bytes(self.automata, aut[a:b], lengths[a:b]) <= ws_bytes // 2
                   for a, b in pairs) or parts >= n:
                return pairs
            parts *= 2

    def call_arrays(self, host_signal, off, lengths, aut, rev, want_seq: bool = True,
                    chunk_reads: int = 25000, lanes: int = 2) -> Dict[str, np.ndarray]:
        """Array-level end-to-end call: (pinned) host signal buffer in, host arrays out --
        len1 ('orig'), len2 ('results'), cost1, cost2, status and, optionally, the decoded
        sequence bytes.  The batch is cut into chunks of up to ``chunk_reads`` reads; one copy
        stream moves the chunks to the device, another brings results back, and the calls
        alternate between ``lanes`` compute streams so that one chunk's kernel tails and
        mid-stage overlap the next chunk's DP.  ``call_batch`` wraps this into ``CallerResult`` objects.

        len/cost/status come back as fresh arrays (-1 / NaN where ``status`` is not 0 -- a read the
        reference would have raised on, see ``_STATUS_ERRORS``); ``seq1``/``seq2`` are views of pinned
        buffers the engine reuses, valid until the next ``call_arrays*`` on it.

        This is the float64 form of the reference's seam (``ReadSignal.signal``, 8 B per sample over
        PCIe); ``call_arrays_quantized`` and ``call_arrays_raw`` take the same reads as int16."""
        lengths = np.asarray(lengths, dtype=np.int32)
        off = np.asarray(off, dtype=np.int64)
        return self._pipeline(_IngestF64(self, host_signal, off, lengths), lengths, aut, rev, want_seq,
                              chunk_reads, lanes)

    def call_arrays_quantized(self, host_raw, raw_off, lengths, host_shift_scale, aut, rev, want_seq: bool = True,
                              chunk_reads: int = 25000, lanes: int = 2) -> Dict[str, np.ndarray]:
        """The same call for reads held as what determines their float64 bits: the int16 samples of each
        window (``host_raw[raw_off[r] : raw_off[r] + lengths[r]]``, after spike removal; pinned; starts on
        multiples of 8 samples for the vector path) and the read's ``{shift, scale}`` (float64 [n, 2], pinned).
        The device evaluates the reference's ``(data - shift) / scale`` (schemas/fast5.py:113) itself
        (wstr_dequantize_batch): a quarter of the bytes cross PCIe and the windows are bit-identical."""
        lengths = np.asarray(lengths, dtype=np.int32)
        raw_off = np.asarray(raw_off, dtype=np.int64)
        return self._pipeline(_IngestI16(self, host_raw, raw_off, lengths, host_shift_scale), lengths, aut, rev,
                              want_seq, chunk_reads, lanes)

    def call_arrays_raw(self, host_raw, raw_off, win_lo, win_hi, aut, rev, spike_removal: str = 'Brute',
                        want_seq: bool = True, chunk_reads: int = 25000, lanes: int = 2) -> Dict[str, np.ndarray]:
        """Raw reads in, calls out (the reference's get_workload -> CallerWrapper.run, wrapper.py:44-54,104-120):
        whole int16 reads ``host_raw[raw_off[r] : raw_off[r+1]]`` and their windows ``[win_lo, win_hi]`` go to
        the device, are spike-filtered, MAD-normalised and sliced there (wstr_normalize_batch) and called
        without the float64 windows ever visiting the host.  The result also carries ``shift_scale``."""
        return self._call_whole(_WholeReads(host_raw, raw_off), win_lo, win_hi, aut, rev, spike_removal, want_seq,
                                chunk_reads, lanes)

    def call_arrays_vbz(self, host_payload, table, read_chunk, raw_off, win_lo, win_hi, aut, rev,
                        spike_removal: str = 'Brute', want_seq: bool = True, chunk_reads: int = 25000,
                        lanes: int = 2) -> Dict[str, np.ndarray]:
        """``call_arrays_raw`` for reads still VBZ-compressed as their fast5 file stores them (``pack_vbz`` makes
        the arguments): only the chunk bodies (after zstd, ~1.25 B per sample instead of 2) cross PCIe, and the
        StreamVByte / zig-zag delta decode (wstr_vbz_decode_batch) writes the int16 reads on the device.  Same
        result dict, plus ``chunk_status`` (WSTR_VBZ_* per chunk) and ``zstd_status`` (WSTR_ZSTD_* per chunk, 0
        for a chunk that was not a zstd frame); a read with a bad chunk has undefined results."""
        return self._call_whole(_VBZReads(host_payload, table, read_chunk, raw_off), win_lo, win_hi, aut, rev,
                                spike_removal, want_seq, chunk_reads, lanes)

    def _call_whole(self, src, win_lo, win_hi, aut, rev, spike_removal, want_seq=True, chunk_reads=25000,
                    lanes=2) -> Dict[str, np.ndarray]:
        """``call_arrays_raw`` of whole reads in any form (a ``_WholeReads``)."""
        from .normalize import SPIKE_MODES
        lo, hi, lengths = _window_bounds(src.raw_off, win_lo, win_hi)
        return self._pipeline(_IngestRaw(self, src, lo, hi, lengths, SPIKE_MODES[spike_removal]), lengths, aut, rev,
                              want_seq, chunk_reads, lanes)

    def _pipeline(self, ingest, lengths, aut, rev, want_seq, chunk_reads, lanes) -> Dict[str, np.ndarray]:
        import torch
        n = len(lengths)
        aut = np.asarray(aut, dtype=np.int32)
        rev = np.asarray(rev, dtype=np.uint8)
        off = ingest.sig_off                                    # float64 windows on the device: even starts
        bounds = self._chunk_bounds(n, max(1, chunk_reads))
        cap = lengths.astype(np.int64) // max(self.cc.min_values_per_state - 1, 1) + 16
        seq_off = np.zeros(n + 1, dtype=np.int64)
        seq_off[1:] = np.cumsum(cap)
        with torch.cuda.device(self.device):
            comp = torch.cuda.current_stream()
            cs_in, cs_out = self._side_streams('copy')
            # signal and result buffers (device, and pinned on the host) live on the engine and only ever grow,
            # so the chunk loop makes no allocator calls
            ingest.allocate()
            d_sig = ingest.d_sig
            buffers = [(k, n, torch.float64 if k in ('cost1', 'cost2') else torch.int32) for k in _SCALARS]
            if want_seq:
                buffers += [(k, int(seq_off[-1]), torch.uint8) for k in ('seq1', 'seq2')]
            dev = {k: self._device_buffer(k, size, dt) for k, size, dt in buffers}
            out = {k: self._host_buffer(k, size, dt) for k, size, dt in buffers}
            cs_in.wait_stream(comp)
            cs_out.wait_stream(comp)
            chunks = list(zip(bounds[:-1], bounds[1:]))

            def mark(label, stream):
                if self.timeline is not None:
                    e = torch.cuda.Event(enable_timing=True)
                    e.record(stream)
                    self.timeline.append((label, e))

            mark('start', comp)

            def send(a, b):                                     # chunk [a, b) -> device, on the input stream
                with torch.cuda.stream(cs_in):
                    mark(f'h2d{a} begin', cs_in)
                    ingest.send(a, b)
                    mark(f'h2d{a} end', cs_in)
                    ev = torch.cuda.Event()
                    ev.record(cs_in)
                return ev

            keep = []
            # every chunk's copy is queued up front (the calls stage their metadata through a
            # kernel, so nothing of theirs waits behind these copies on the DMA engine); the
            # host only has to keep the compute stream fed
            h2d_begin = torch.cuda.Event(enable_timing=True)
            h2d_begin.record(cs_in)
            sent = [send(a, b) for a, b in chunks]
            h2d_end = torch.cuda.Event(enable_timing=True)
            h2d_end.record(cs_in)
            if ingest.h2d_bytes:        # (reads already on the device say nothing about the host link)
                self._h2d_probe = (h2d_begin, h2d_end, int(ingest.h2d_bytes))
            # chunks alternate between `lanes` compute streams (each with its own workspace): the
            # kernels of consecutive chunks are independent, so one chunk's kernel tails and
            # latency-bound mid-stage overlap the next chunk's DP
            n_lanes = max(1, int(lanes))
            streams = [comp] + (self._side_streams('lanes')[:n_lanes - 1] if n_lanes > 1 else [])
            for st in streams[1:]:
                st.wait_stream(comp)
            for ci, (a, b) in enumerate(chunks):
                ev = sent[ci]
                lane = ci % len(streams)
                st = streams[lane]
                lo, hi = _span(off, lengths, a, b, d_sig.numel())
                with torch.cuda.stream(st):
                    st.wait_event(ev)
                    mark(f'call{a} begin', st)
                    ingest.prepare(a, b, lane)                  # int16 forms: the float64 windows are made here
                    into = {k: dev[k][a:b] for k in _SCALARS}
                    if want_seq:
                        into['seq1'] = dev['seq1'][int(seq_off[a]):int(seq_off[b])]
                        into['seq2'] = dev['seq2'][int(seq_off[a]):int(seq_off[b])]
                    o = self.call_packed(d_sig[lo:hi], off[a:b] - lo, lengths[a:b], aut[a:b], rev[a:b],
                                         want_seq=want_seq, into=into, lane=lane, allow_split=False)
                    mark(f'call{a} end', st)
                    done = torch.cuda.Event()
                    done.record(st)
                with torch.cuda.stream(cs_out):                 # results back while the next chunk computes
                    cs_out.wait_event(done)
                    for k in _SCALARS:
                        out[k][a:b].copy_(o[k], non_blocking=True)
                    if want_seq:
                        s0, s1 = int(seq_off[a]), int(seq_off[b])
                        out['seq1'][s0:s1].copy_(o['seq1'][:s1 - s0], non_blocking=True)
                        out['seq2'][s0:s1].copy_(o['seq2'][:s1 - s0], non_blocking=True)
                    ingest.fetch(a, b)
                    mark(f'd2h{a} end', cs_out)
                keep.append(o)
            for st in streams[1:]:
                comp.wait_stream(st)
            cs_out.synchronize()
            comp.wait_stream(cs_in)
            comp.wait_stream(cs_out)
        # per-read scalars are handed back as copies; reads the device could not finish (status != 0) carry
        # -1 / NaN instead of whatever the buffers held.  The sequence bytes are views of the engine's pinned
        # buffers (hundreds of MB per 100 000 reads): valid until the next call_arrays on this engine.
        res = {k: out[k].numpy().copy() for k in _SCALARS}
        res['ttest_ties'] = res.pop('ties')
        bad = res['status'] != 0
        if bad.any():
            res['len1'][bad] = -1
            res['len2'][bad] = -1
            res['cost1'][bad] = np.nan
            res['cost2'][bad] = np.nan
        if want_seq:
            res['seq1'] = out['seq1'].numpy()
            res['seq2'] = out['seq2'].numpy()
            res['seq_off'] = seq_off[:-1]
        ingest.finish(res)
        return res

    def _chunk_bounds(self, n: int, step: int):
        """Chunk boundaries of the end-to-end pipeline.  The first chunk is short (its copy is the
        only one nothing overlaps) and sizes double from there.  When the host link keeps well
        ahead of the kernels (one GPU per host link: ~55 GB/s measured) they double up to ``step``;
        when the previous call's copies ran slower (several GPUs sharing the host's memory
        system) chunks stay small and shrink again at the end, because then the time after the last
        copy -- one chunk's worth of kernels -- is what is exposed."""
        slow_link = False
        probe = self._h2d_probe
        if probe is not None and probe[1].query():
            ms = probe[0].elapsed_time(probe[1])
            slow_link = ms > 0 and probe[2] / ms / 1e6 < 40.0        # GB/s
        first = max(1, step // 8)
        if not slow_link:
            bounds, size = [0], first
            while bounds[-1] < n:
                bounds.append(min(n, bounds[-1] + size))
                size = min(step, size * 2)
            return bounds
        cap = max(first, step // 2)
        up, size, used = [], first, 0
        while size < cap and used + 2 * size <= n:                     # mirrored ramps at both ends
            up.append(size)
            used += 2 * size
            size *= 2
        mid = n - used
        sizes = list(up)
        while mid > 0:
            take = min(cap, mid)
            sizes.append(take)
            mid -= take
        sizes += up[::-1]
        bounds = [0]
        for sz in sizes:
            bounds.append(bounds[-1] + sz)
        return bounds

    def _device_buffer(self, name: str, numel: int, dtype):
        import torch
        cur = self._dev_cache.get(name)
        if cur is None or cur.numel() < numel or cur.dtype != dtype:
            self._dev_cache[name] = None
            cur = torch.empty(max(numel, 1), dtype=dtype, device=self.device)
            self._dev_cache[name] = cur
        return cur[:numel]

    def _host_buffer(self, name: str, numel: int, dtype):
        """Pinned host buffer ``name`` as ``_device_buffer`` keeps device ones: grown on demand and reused."""
        import torch
        cur = self._host_cache.get(name)
        if cur is None or cur.numel() < numel or cur.dtype != dtype:
            cur = torch.empty(max(numel, 1), dtype=dtype, pin_memory=torch.cuda.is_available())
            self._host_cache[name] = cur
        return cur[:numel]

    def call_raw_batch(self, raws: Sequence[np.ndarray], windows, aut_ids, reverse,
                       spike_removal: str = 'Brute', offset: float = 0.35) -> list:
        """Raw int16 reads and their STR windows in, CallerResults out: the reference's
        ``get_workload`` + ``CallerWrapper.run`` (wrapper.py:44-54, 104-120) as one device-resident chain
        (``call_arrays_raw``: normalisation kernel -> caller, the float64 windows never leave the GPU).

        ``windows=None``: the windows are found first, in the whole reads, by ``locate_arrays_raw`` (score offset
        ``offset``); the int16 reads stay on the device for the call.  A read whose window is not found is
        not called: its entry is a ``NotLocated``.  The located windows are in ``last_located``.  Here an entry
        of ``aut_ids`` may be a (template id, reverse id) pair (its ``reverse`` entry is ignored, e.g. None): the
        read is searched on both strands and called with the strand ``choose_strand`` picks, whose id and
        orientation are then used; ``last_located['strand']`` has every read's strand, given or detected."""
        if len(raws) == 0:
            return []
        src = _WholeReads(*pack_raw(raws), samples=lambda idx: [raws[r] for r in idx])
        return self._call_reads(src, windows, aut_ids, reverse, spike_removal, offset)

    def call_vbz_batch(self, reads, windows, aut_ids, reverse, spike_removal: str = 'Brute',
                       offset: float = 0.35) -> list:
        """``call_raw_batch`` for reads as their fast5 files store them (fast5.CompressedRead, from
        ``fast5.raw_chunks``): the chunk bodies go to the device, are decoded there (wstr_vbz_decode_batch) and
        called as ``call_raw_batch`` calls raw reads.  A chunk the host decoder would refuse raises that
        Fast5FormatError, naming the file and the read, before any result is returned.  ``windows=None``
        locates the windows first (``locate_arrays_vbz``): the payload crosses PCIe once and the decoded reads
        stay on the device for the call; reads not found come back as ``NotLocated``.  Strand pairs in ``aut_ids``
        as in ``call_raw_batch``."""
        if len(reads) == 0:
            return []
        if any(r.n_samples <= 0 for r in reads):
            raise ValueError('empty raw read')
        return self._call_reads(_VBZReads(*pack_vbz(reads), reads), windows, aut_ids, reverse, spike_removal, offset)

    def _call_reads(self, src, windows, aut_ids, reverse, spike_removal, offset) -> list:
        """``call_raw_batch`` of whole reads in any form (a ``_WholeReads``)."""
        if windows is None:
            return self._call_located(src, aut_ids, reverse, spike_removal, offset)
        res = self._call_whole(src, [w[0] for w in windows], [w[1] for w in windows], _single_ids(aut_ids),
                               np.asarray(reverse, dtype=np.uint8), spike_removal)
        src.raise_bad(res)

        def signals_of(idx):
            from .normalize import normalize_windows
            return normalize_windows(src.samples(idx), [windows[r] for r in idx], spike_removal,
                                     device=str(self.device))
        return self._results(res, signals_of, aut_ids, reverse)

    # -- STR window search in whole reads (DESIGN.md section 4.5) ----------------------------------------------
    def locate_packed(self, d_sig, off, lengths, aut, offset: float = 0.35) -> Dict[str, np.ndarray]:
        """wstr_locate_batch on device-resident whole normalised reads (float64, even starts ``off``).  Returns
        host arrays: ``lo``, ``hi`` (the window, inclusive, in the read's samples), ``score`` and ``status``
        (_lib.LOCATE_*: found iff the score is below zero).

        ``aut[r]`` is one automaton id, or a (template id, reverse id) pair for a read whose strand is not known.
        Such a read enters the launch twice, both entries on the same samples, one after the other (the plan's
        stable longest-first order keeps them adjacent, so both CTAs read the read while it is in L2), and
        ``choose_strand`` decides: ``lo``, ``hi``, ``score``, ``status`` are the chosen strand's, ``strand`` is
        0 (template), 1 (reverse) or -1 (found on neither), and ``strand_score`` (float64[n, 2]),
        ``strand_status``, ``strand_lo``, ``strand_hi`` (int32[n, 2]) hold both searches.  A read given one id
        has NaN / -1 there and ``strand`` -1: which strand its automaton is is the caller's to say
        (``fill_given_strands``)."""
        import torch
        n = len(lengths)
        lengths = np.asarray(lengths, dtype=np.int32)
        off = np.asarray(off, dtype=np.int64)
        pair, ids = split_pairs(aut)
        reps = 1 + pair.astype(np.int64)
        first = np.cumsum(reps) - reps                       # each read's first entry
        entry_read = np.repeat(np.arange(n), reps)
        entry_aut = ids[entry_read, np.arange(len(entry_read)) - first[entry_read]]
        m = len(entry_read)
        with torch.cuda.device(self.device):
            ws = self._device_buffer('loc_ws', _lib.locate_workspace_bytes(self.automata, m), torch.uint8)
            d_i = torch.empty((3, max(m, 1)), dtype=torch.int32, device=self.device)
            d_score = torch.empty(max(m, 1), dtype=torch.float64, device=self.device)
            _lib.locate_batch(self.automata, entry_aut, d_sig, off[entry_read], lengths[entry_read], offset,
                              d_i[0], d_i[1], d_score, d_i[2], ws)
            h_i = d_i.cpu().numpy()
            e_score = d_score.cpu().numpy()
        second = first + pair
        st2 = np.stack((h_i[2, first], h_i[2, second]), axis=1)
        sc2 = np.stack((e_score[first], e_score[second]), axis=1)
        strand, col, status, score = choose_strand(st2, sc2)     # a single entry is its own "pair": unchanged
        pick = np.where(col == 1, second, first)
        lo2 = np.stack((h_i[0, first], h_i[0, second]), axis=1)
        hi2 = np.stack((h_i[1, first], h_i[1, second]), axis=1)
        strand[~pair] = -1
        for a in (st2, lo2, hi2):
            a[~pair] = -1
        sc2[~pair] = np.nan
        return dict(lo=h_i[0, pick], hi=h_i[1, pick], score=score, status=status, strand=strand,
                    strand_score=sc2, strand_status=st2, strand_lo=lo2, strand_hi=hi2)

    def locate_arrays_raw(self, host_raw, raw_off, aut, spike_removal: str = 'Brute',
                          offset: float = 0.35) -> Dict[str, np.ndarray]:
        """Whole int16 reads ``host_raw[raw_off[r] : raw_off[r+1]]`` (``pack_raw``) in, their STR windows out:
        whole-read normalisation (wstr_normalize_batch, window [0, N-1]) and the window search on the device.
        ``aut`` and the dict as in ``locate_packed``."""
        return self._locate_whole(_WholeReads(host_raw, raw_off), aut, spike_removal, offset)

    def locate_arrays_vbz(self, host_payload, table, read_chunk, raw_off, aut, spike_removal: str = 'Brute',
                          offset: float = 0.35) -> Dict[str, np.ndarray]:
        """``locate_arrays_raw`` for VBZ-compressed reads (``pack_vbz``): decoded on the device first.  The dict
        also carries ``chunk_status`` (WSTR_VBZ_* per chunk) and ``zstd_status`` (WSTR_ZSTD_* per chunk); a read
        with a bad chunk has undefined results."""
        return self._locate_whole(_VBZReads(host_payload, table, read_chunk, raw_off), aut, spike_removal, offset)

    def _locate_whole(self, src, aut, spike_removal, offset) -> Dict[str, np.ndarray]:
        """``locate_arrays_raw`` of whole reads in any form (a ``_WholeReads``), with its decode statuses."""
        st = self._load(src)
        res = self._locate_device(src.d_raw, src.raw_off, aut, spike_removal, offset)
        res.update(st)
        return res

    def _load(self, src) -> dict:
        """Every read of ``src`` sent and decoded on the current stream into the device buffer 'loc_raw16' (which
        the pipelined call does not grow or write, so located reads can be called from it); returns the decode
        statuses as ``finish`` puts them into a result."""
        import torch
        n = len(src.raw_off) - 1
        with torch.cuda.device(self.device):
            src.allocate(self, 'loc_raw16')
            src.send(0, n)
            src.decode(self, 0, n, 0)
            src.fetch(0, n)
            torch.cuda.current_stream().synchronize()
        st = {}
        src.finish(st)
        return st

    def _normalize_whole(self, d_raw, raw_off, spike_removal):
        """Whole-read normalisation of int16 reads on the device (window [0, N-1]) for the searches in whole reads:
        (d_sig float64, sig_off, lengths)."""
        import torch
        from .normalize import SPIKE_MODES
        lens = np.diff(raw_off)
        if (lens > _lib.LOCATE_MAX_SAMPLES).any():
            raise ValueError(f'a read longer than {_lib.LOCATE_MAX_SAMPLES} samples cannot be located')
        lengths = lens.astype(np.int32)
        n = len(lengths)
        sig_off, total = even_offsets(lengths)
        with torch.cuda.device(self.device):
            d_sig = torch.empty(total, dtype=torch.float64, device=self.device)
            ws = self._device_buffer('norm_ws0', _lib.normalize_workspace_bytes(n), torch.uint8)
            _lib.normalize_batch(d_raw, raw_off, np.zeros(n, dtype=np.int32), lengths - 1, SPIKE_MODES[spike_removal],
                                 d_sig, sig_off, None, ws)
        return d_sig, sig_off, lengths

    def _locate_device(self, d_raw, raw_off, aut, spike_removal, offset) -> Dict[str, np.ndarray]:
        """Whole-read normalisation of int16 reads on the device, then the window search."""
        import torch
        d_sig, sig_off, lengths = self._normalize_whole(d_raw, raw_off, spike_removal)
        with torch.cuda.device(self.device):
            res = self.locate_packed(d_sig, sig_off, lengths, aut, offset)
            del d_sig
        return res

    # -- a panel's reads found in a whole run by their flanks (DESIGN.md section 4.6) ----------------------------
    def assign_packed(self, d_sig, off, lengths, panel, offset: float = 0.35) -> Dict[str, np.ndarray]:
        """wstr_assign_batch on device-resident whole normalised reads (float64, even starts ``off``) with the flank
        chains of ``panel`` (an ``assign.Panel``; its chains are uploaded to this engine on first use).  Returns the
        hits as host arrays sorted by (read, locus), the fields of ``assign.HIT_FIELDS``: every (read, locus) whose
        flanks were found in order on a strand, and that strand (0 template, 1 reverse).  Only the hits leave the
        device."""
        import torch
        ids = panel.register(self)
        auts = [self.automata[i] for i in ids]
        n = len(lengths)
        cap = max(n * (len(auts) // 4), 1) * _lib.ASSIGN_HIT.itemsize
        with torch.cuda.device(self.device):
            ws = self._device_buffer('asg_ws', _lib.assign_workspace_bytes(auts, n), torch.uint8)
            d_hits = self._device_buffer('asg_hits', cap, torch.uint8)
            d_n = self._device_buffer('asg_n', 1, torch.int32)
            _lib.assign_batch(auts, d_sig, off, lengths, offset, None, d_hits, d_n, ws)
            k = int(d_n.cpu()[0])
            hits = d_hits[:k * _lib.ASSIGN_HIT.itemsize].cpu().numpy().view(_lib.ASSIGN_HIT)
        return hit_arrays(hits)

    def assign_arrays_raw(self, host_raw, raw_off, panel, spike_removal: str = 'Brute',
                          offset: float = 0.35) -> Dict[str, np.ndarray]:
        """Whole int16 reads (``pack_raw``) in, the panel's hits out (``assign_packed``): upload, whole-read
        normalisation and the flank search on the device."""
        return self._assign_whole(_WholeReads(host_raw, raw_off), panel, spike_removal, offset)

    def assign_arrays_vbz(self, host_payload, table, read_chunk, raw_off, panel, spike_removal: str = 'Brute',
                          offset: float = 0.35, reads=None) -> Dict[str, np.ndarray]:
        """``assign_arrays_raw`` for VBZ-compressed reads (``pack_vbz``), decoded on the device first.  With
        ``reads`` (the fast5.CompressedRead list packed) a chunk the device decoders refuse raises its
        Fast5FormatError, naming the file and the read; without, the dict carries ``chunk_status`` and
        ``zstd_status`` and a read with a bad chunk has undefined hits."""
        src = _VBZReads(host_payload, table, read_chunk, raw_off, reads)
        res = self._assign_whole(src, panel, spike_removal, offset)
        if reads is not None:
            src.raise_bad(res)
        return res

    def _assign_whole(self, src, panel, spike_removal, offset) -> Dict[str, np.ndarray]:
        import torch
        st = self._load(src)
        d_sig, sig_off, lengths = self._normalize_whole(src.d_raw, src.raw_off, spike_removal)
        with torch.cuda.device(self.device):
            res = self.assign_packed(d_sig, sig_off, lengths, panel, offset)
            del d_sig
        res.update(st)
        return res

    def _call_located(self, src, aut_ids, reverse, spike_removal, offset) -> list:
        """The located-then-called chain: send and decode the whole reads, locate, bring the windows to the
        host, normalise the found windows and call them from the same device buffer, each with the automaton
        and orientation of its strand (given, or chosen by the both-strand search)."""
        import torch
        src.raise_bad(self._load(src))
        d_raw, raw_off = src.d_raw, src.raw_off
        loc = self._locate_device(d_raw, raw_off, aut_ids, spike_removal, offset)
        pair, ids = split_pairs(aut_ids)
        fill_given_strands(loc, [None if p else r for p, r in zip(pair, reverse)])
        self.last_located = loc
        rev = loc['strand'].clip(0, 1).astype(np.uint8)
        aut = ids[np.arange(len(rev)), rev]
        out: list = [NotLocated(int(st), float(sc)) for st, sc in zip(loc['status'], loc['score'])]
        found = np.flatnonzero(loc['status'] == _lib.LOCATE_FOUND)
        if not len(found):
            return out
        if len(found) < len(out):         # the found reads, packed
            with torch.cuda.device(self.device):
                d_raw = torch.cat([d_raw[int(raw_off[r]):int(raw_off[r + 1])] for r in found])
            raw_off = np.zeros(len(found) + 1, dtype=np.int64)
            raw_off[1:] = np.cumsum(np.diff(src.raw_off)[found])
        located = _WholeReads(None, raw_off, d_raw, samples=lambda idx: src.samples([int(found[k]) for k in idx]))
        windows = list(zip(loc['lo'][found].tolist(), loc['hi'][found].tolist()))
        calls = self._call_reads(located, windows, aut[found], rev[found], spike_removal, offset)
        for k, r in enumerate(found):
            out[r] = calls[k]
        return out

    def results_from(self, o, signals, aut_ids, reverse) -> List[CallerResult]:
        """Device results -> CallerResult list; reads the device could not finish (status != 0)
        are redone on the host path or raise what the reference raises."""
        h = {k: o[k].cpu().numpy() for k in ('status', 'ties', 'len1', 'len2', 'cost1', 'cost2', 'seq1', 'seq2')
             if k in o}
        h['ttest_ties'] = h.pop('ties', np.zeros_like(h['status']))
        return self._results(dict(h, seq_off=o['seq_off']), lambda idx: [signals[r] for r in idx], aut_ids, reverse)

    def _results(self, h, signals_of, aut_ids, reverse) -> List[CallerResult]:
        """CallerResults of the host result arrays ``h`` of a call (as ``call_arrays`` returns them).  Reads the
        device did not finish (status != 0), or whose t-test decision was within rounding of flipping (ttest_ties
        > 0), are redone on the host path from their float64 windows, ``signals_of(indices)``."""
        status, ties, len1, len2, cost1, cost2, seq1, seq2, off = (
            h[k] for k in ('status', 'ttest_ties', 'len1', 'len2', 'cost1', 'cost2', 'seq1', 'seq2', 'seq_off'))
        self.last_ttest_ties = int((ties > 0).sum())
        out: List[Optional[CallerResult]] = []
        redo = []
        for r in range(len(status)):
            # (a read with a t-test decision within rounding distance of flipping is decided by the libm the
            # reference runs on -- np.float64 ** 2 is pow(), caller.py:351 -- so it is evaluated on the host)
            if status[r] == 0 and ties[r] == 0:
                a = int(off[r])
                out.append(CallerResult(seq=seq1[a:a + len1[r]].tobytes().decode('ascii'), cost=float(cost1[r]),
                                        resc_seq=seq2[a:a + len2[r]].tobytes().decode('ascii'),
                                        resc_cost=float(cost2[r])))
            else:
                out.append(None)
                redo.append(r)
        if redo:
            # status 5 (spline needs interior knots) is a legitimate host evaluation; every other
            # status is an exception in the reference, which the host path raises with its type
            fixed = self._call_batch_host(signals_of(redo), [aut_ids[r] for r in redo], [reverse[r] for r in redo])
            for r, res in zip(redo, fixed):
                out[r] = res
        return out

    def _call_batch_host(self, signals, aut_ids, reverse) -> List[CallerResult]:
        """Both DP passes on the GPU, the stage between them with the reference's own numpy/scipy
        calls on the host.  Never silent: used for ``reps_as_one``, for reads whose smoothing spline
        needs interior knots (impossible at the default thresholds) and to raise the reference's
        exception for a read the device flagged."""
        import warnings
        warnings.warn(f'warpstr_b200: {len(signals)} read(s) take the host mid-stage (scipy splrep/splev); '
                      'the DP passes still run on the GPU', RuntimeWarning, stacklevel=3)
        traces1 = self.warp_batch(signals, aut_ids)
        first = []
        for s, a, t in zip(signals, aut_ids, traces1):
            tb = self.tables[a]
            first.append(self._after(t, s, tb, False))
        traces2 = self.warp_batch([p.rescaled for p in first], aut_ids, [p.badmask for p in first])
        out = []
        for p1, a, t2, rev in zip(first, aut_ids, traces2, reverse):
            tb = self.tables[a]
            p2 = self._after(t2, p1.rescaled, tb, True)
            out.append(CallerResult(seq=self.decode(a, p1.runs, rev), cost=p1.cost,
                                    resc_seq=self.decode(a, p2.runs, rev), resc_cost=p2.cost))
        return out

    def _after(self, trace, x, tb, second):
        try:
            return midstage.after_pass(trace, x, tb['values'], tb['rep_mask'], self.cc, self.rc, second)
        except midstage.ReadError as e:
            raise e.kind(str(e))


def _single_ids(aut_ids) -> np.ndarray:
    """Automaton ids of reads called on given windows: one per read, a strand pair is refused (the strand is not
    searched inside a given window)."""
    pair, ids = split_pairs(aut_ids)
    if pair.any():
        raise ValueError(f'read {int(np.flatnonzero(pair)[0])} of the batch: a given window needs a given strand '
                         '(one automaton id, not a pair)')
    return ids[:, 0].copy()


_default_engine: Optional[CallerEngine] = None


def default_engine(caller_config=None, rescaler_config=None) -> CallerEngine:
    global _default_engine
    if _default_engine is None or caller_config is not None or rescaler_config is not None:
        _default_engine = CallerEngine(caller_config, rescaler_config)
    return _default_engine


class _StatesView:
    """Flat tables out of a list of State-like objects (kmer, value, seq_idx, idx, incoming)."""

    def __init__(self, states, endstate, repeat_mask):
        S = len(states)
        self.values = np.array([s.value for s in states], dtype=np.float64)
        self.seq_idx = np.array([s.seq_idx for s in states], dtype=np.int32)
        self.in_ptr = np.zeros(S + 1, dtype=np.int32)
        idx: List[int] = []
        for i, s in enumerate(states):
            idx.extend(p.idx for p in s.incoming)
            self.in_ptr[i + 1] = len(idx)
        self.in_idx = np.array(idx, dtype=np.int32)
        self.rep_mask = np.array(repeat_mask, dtype=np.uint8)
        self.last_base = np.frombuffer(''.join(s.kmer[-1] for s in states).encode('ascii'), dtype=np.uint8).copy()
        self.endstate = int(endstate)


@dataclass
class WarpSTR:
    """Single-read seam with the reference's constructor (caller.py:107-115)."""
    flank_length: int
    states: list
    endstate: int
    repeat_mask: List[bool]
    out_warp_path: Optional[str]
    reverse: bool
    read_name: str
    engine: Optional[CallerEngine] = None

    def __post_init__(self):
        self._engine = self.engine or default_engine()
        # the reference builds one WarpSTR per read from the locus's automaton (wrapper.py:289,329): the
        # uploaded tables are shared between them, keyed on their content (ids of Python objects can be
        # recycled once a locus's automaton has been collected)
        view = _StatesView(self.states, self.endstate, self.repeat_mask)
        key = hashlib.sha1(b''.join(a.tobytes() for a in (view.values, view.seq_idx, view.in_ptr, view.in_idx,
                                                            view.rep_mask, view.last_base)) +
                           repr((view.endstate, int(self.flank_length),
                                 int(self._engine.cc.min_values_per_state))).encode()).hexdigest()
        cache = self._engine.__dict__.setdefault('_seam_cache', {})
        if key not in cache:
            if len(cache) >= 64:                       # a long run over many loci: drop the oldest upload
                cache.pop(next(iter(cache)))
            cache[key] = self._engine.add_automaton(view, self.flank_length)
        self._aut = cache[key]

    def warp(self, signal: np.ndarray, mask: Optional[List[bool]] = None) -> WarpResult:
        sig = np.ascontiguousarray(signal, dtype=np.float64)
        use_mask = mask is not None and len(mask) > 0
        traces = self._engine.warp_batch([sig], [self._aut], [np.asarray(mask, dtype=bool)] if use_mask else None)
        return WarpResult(traces[0].astype(int))

    def run(self, signal: np.ndarray) -> CallerResult:
        return self._engine.call_batch([signal], [self._aut], [self.reverse])[0]
