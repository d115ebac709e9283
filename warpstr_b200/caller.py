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
    padded = (lengths.astype(np.int64) + 1) & ~1
    offsets = np.zeros(n, dtype=np.int64)
    if n > 1:
        offsets[1:] = np.cumsum(padded[:-1])
    total = int(padded.sum()) + 2
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


class _IngestF64:
    """Host float64 windows (the reference's ReadSignal.signal): copied as they are."""

    def __init__(self, eng, host_signal, off, lengths):
        self.eng, self.host, self.sig_off, self.lengths = eng, host_signal, off, lengths
        n = len(lengths)
        self.total = int(off[-1] + ((int(lengths[-1]) + 1) & ~1) + 2) if n else 0
        self.h2d_bytes = min(self.total, host_signal.numel()) * 8

    def allocate(self):
        import torch
        self.d_sig = self.eng._device_buffer('sig', min(self.total, self.host.numel()), torch.float64)

    def send(self, a, b):
        lo = int(self.sig_off[a])
        hi = min(int(self.sig_off[b - 1] + ((int(self.lengths[b - 1]) + 1) & ~1) + 2), self.d_sig.numel())
        self.d_sig[lo:hi].copy_(self.host[lo:hi], non_blocking=True)

    def prepare(self, a, b, lane):
        pass

    def fetch(self, a, b, out):
        pass

    def finish(self, res, out, n):
        pass


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

    def fetch(self, a, b, out):
        pass

    def finish(self, res, out, n):
        pass


class _IngestRaw:
    """Host int16 whole reads + windows; spike removal, MAD normalisation and slicing on the device."""

    def __init__(self, eng, host_raw, raw_off, lo, hi, lengths, spike_mode):
        self.eng, self.host, self.raw_off, self.lo, self.hi = eng, host_raw, raw_off, lo, hi
        self.lengths, self.spike_mode = lengths, spike_mode
        self.sig_off, self.total = even_offsets(lengths)
        self.h2d_bytes = int(raw_off[-1]) * 2 if len(raw_off) else 0
        self.d_raw = None

    def allocate(self):
        import torch
        e = self.eng
        self.d_sig = e._device_buffer('sig', self.total, torch.float64)
        if self.d_raw is None:
            self.d_raw = e._device_buffer('raw16', int(self.raw_off[-1]), torch.int16)
        self.d_ss = e._device_buffer('shift_scale', 2 * len(self.lengths), torch.float64)
        pin = torch.cuda.is_available()
        cur = e._host_ss
        if cur is None or cur.numel() < 2 * len(self.lengths):
            e._host_ss = torch.empty(max(2 * len(self.lengths), 2), dtype=torch.float64, pin_memory=pin)

    def send(self, a, b):
        lo, hi = int(self.raw_off[a]), int(self.raw_off[b])
        self.d_raw[lo:hi].copy_(self.host[lo:hi], non_blocking=True)

    def prepare(self, a, b, lane):
        import torch
        n = b - a
        ws = self.eng._device_buffer(f'norm_ws{lane}', _lib.normalize_workspace_bytes(n), torch.uint8)
        _lib.normalize_batch(self.d_raw, self.raw_off[a:b + 1], self.lo[a:b], self.hi[a:b], self.spike_mode,
                             self.d_sig, self.sig_off[a:b], self.d_ss[2 * a:2 * b], ws)

    def fetch(self, a, b, out):
        self.eng._host_ss[2 * a:2 * b].copy_(self.d_ss[2 * a:2 * b], non_blocking=True)

    def finish(self, res, out, n):
        res['shift_scale'] = self.eng._host_ss[:2 * n].numpy().reshape(n, 2).copy()
        res['lengths'] = self.lengths


class _IngestDeviceRaw(_IngestRaw):
    """Whole int16 reads that are already on the device (the located-then-called chain): nothing crosses
    PCIe, the windows are normalised and called as in _IngestRaw."""

    def __init__(self, eng, d_raw, raw_off, lo, hi, lengths, spike_mode):
        super().__init__(eng, None, raw_off, lo, hi, lengths, spike_mode)
        self.d_raw = d_raw
        self.h2d_bytes = 0

    def send(self, a, b):
        pass


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
    buffer (every chunk's body at a 16-byte aligned offset, zero padded: the decoder reads whole 16-byte
    words), the chunk table, the first chunk of every read (int64[n + 1]) and the read offsets in the
    decoded int16 buffer (int64[n + 1])."""
    import torch
    chunks = [c for r in reads for c in r.chunks]
    m = len(chunks)
    n_chunks = np.fromiter((len(r.chunks) for r in reads), dtype=np.int64, count=len(reads))
    read_chunk = np.zeros(len(reads) + 1, dtype=np.int64)
    read_chunk[1:] = np.cumsum(n_chunks)
    raw_off = np.zeros(len(reads) + 1, dtype=np.int64)
    raw_off[1:] = np.cumsum(np.fromiter((r.n_samples for r in reads), dtype=np.int64, count=len(reads)))
    in_bytes = np.fromiter((len(c.payload) for c in chunks), dtype=np.int64, count=m)
    in_off = np.zeros(m + 1, dtype=np.int64)
    in_off[1:] = np.cumsum((in_bytes + 15) & ~15)
    chunk_read = np.repeat(np.arange(len(reads)), n_chunks)
    table = dict(in_off=in_off[:-1], in_bytes=in_bytes,
                 n_samples=np.fromiter((c.coded if c.kind != 2 else c.count for c in chunks), dtype=np.int32, count=m),
                 n_out=np.fromiter((c.count for c in chunks), dtype=np.int32, count=m),
                 kind=np.fromiter((c.kind for c in chunks), dtype=np.int32, count=m),
                 zigzag=np.fromiter((c.zigzag for c in chunks), dtype=np.int32, count=m),
                 out_off=raw_off[chunk_read] + np.fromiter((c.start for c in chunks), dtype=np.int64, count=m))
    host = torch.zeros(max(int(in_off[-1]), 16), dtype=torch.uint8, pin_memory=torch.cuda.is_available())
    hb = host.numpy()
    for c, o in zip(chunks, in_off[:-1]):
        hb[o:o + len(c.payload)] = np.frombuffer(c.payload, dtype=np.uint8)
    return host, table, read_chunk, raw_off


class _IngestVBZ(_IngestRaw):
    """VBZ chunk bodies (after zstd) of whole reads + windows: the StreamVByte / delta decode
    (wstr_vbz_decode_batch) writes the int16 reads on the device, which then go on as in _IngestRaw."""

    def __init__(self, eng, host_payload, table, read_chunk, raw_off, lo, hi, lengths, spike_mode):
        super().__init__(eng, None, raw_off, lo, hi, lengths, spike_mode)
        self.payload, self.table, self.read_chunk = host_payload, table, read_chunk
        m = len(table['in_off'])
        self.pay_off = np.append(table['in_off'], int(table['in_off'][-1] + ((table['in_bytes'][-1] + 15) & ~15))
                                 if m else 0)[read_chunk]                     # payload bytes of reads [a, b)
        self.h2d_bytes = int(self.pay_off[-1]) if len(self.pay_off) else 0

    def allocate(self):
        import torch
        super().allocate()
        e = self.eng
        m = len(self.table['in_off'])
        self.d_payload = e._device_buffer('vbz_payload', max(self.h2d_bytes, 16), torch.uint8)
        self.d_status = e._device_buffer('vbz_status', m, torch.int32)
        cur = e._host_vbz_status
        if cur is None or cur.numel() < m:
            e._host_vbz_status = torch.empty(max(m, 1), dtype=torch.int32, pin_memory=torch.cuda.is_available())

    def send(self, a, b):
        lo, hi = int(self.pay_off[a]), int(self.pay_off[b])
        self.d_payload[lo:hi].copy_(self.payload[lo:hi], non_blocking=True)

    def prepare(self, a, b, lane):
        import torch
        c0, c1 = int(self.read_chunk[a]), int(self.read_chunk[b])
        if c1 > c0:
            t = {k: v[c0:c1] for k, v in self.table.items()}
            ws = self.eng._device_buffer(f'vbz_ws{lane}', _lib.vbz_workspace_bytes(c1 - c0), torch.uint8)
            _lib.vbz_decode_batch(self.d_payload, t['in_off'], t['in_bytes'], t['n_samples'], t['n_out'], t['kind'],
                                  t['zigzag'], t['out_off'], self.d_raw, self.d_status[c0:c1], ws)
        super().prepare(a, b, lane)

    def fetch(self, a, b, out):
        super().fetch(a, b, out)
        c0, c1 = int(self.read_chunk[a]), int(self.read_chunk[b])
        self.eng._host_vbz_status[c0:c1].copy_(self.d_status[c0:c1], non_blocking=True)

    def finish(self, res, out, n):
        super().finish(res, out, n)
        res['chunk_status'] = self.eng._host_vbz_status[:len(self.table['in_off'])].numpy().copy()


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
        self._ws = None
        self._ws_at_limit = False
        self._ws_need_seen = 0
        self._lane_ws = {}
        self._lane_streams = None
        self._copy_stream = None
        self.timeline = None      # set to a list to collect (label, CUDA event) pairs from call_arrays
        self._host_out = None
        self._host_ss = None
        self._host_vbz_status = None
        self._dev_cache = {}
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
        if lane:
            # extra compute lanes of the pipelined call own a workspace each (sized for their chunks), under
            # the same limits as the first: the explicit one, else 60 % of what is free when it has to grow
            ws = self._lane_ws.get(lane)
            if ws is None or ws.numel() < need:
                import torch
                have = ws.numel() if ws is not None else 0
                limit = self.workspace_limit
                if limit is None:
                    free, _ = torch.cuda.mem_get_info(self.device)
                    limit = int(free * 0.6) + have
                size = min(need, max(limit, 1 << 20))
                if size > have:
                    self._lane_ws[lane] = None
                    ws = torch.empty(size, dtype=torch.uint8, device=self.device)
                    self._lane_ws[lane] = ws
            return ws
        return self._workspace0(need)

    def _workspace0(self, need: int):
        """Device workspace of ``need`` bytes, or as much as the memory limit allows (the library
        then works in waves).  The buffer only grows; cudaMemGetInfo is asked only when it has
        to (the call can block for tens of milliseconds while the GPU is busy)."""
        import torch
        ws = self._ws
        if ws is not None and (ws.numel() >= need or (self._ws_at_limit and need <= self._ws_need_seen)):
            return ws
        self._ws_need_seen = need        # a larger request re-evaluates the limit (memory may have been freed)
        limit = self.workspace_limit
        if limit is None:
            free, _ = torch.cuda.mem_get_info(self.device)
            limit = int(free * 0.6) + (ws.numel() if ws is not None else 0)
        size = min(need, max(limit, 1 << 20))
        self._ws_at_limit = size < need
        if ws is None or ws.numel() < size:
            self._ws = None
            self._ws = torch.empty(size, dtype=torch.uint8, device=self.device)
        return self._ws

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
                    o['seq1'] = torch.empty(total, dtype=torch.uint8, device=self.device)
                    o['seq2'] = torch.empty(total, dtype=torch.uint8, device=self.device)
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
                lo = int(off[a])
                hi = min(int(off[b - 1] + ((int(lengths[b - 1]) + 1) & ~1) + 2), d_sig.numel()) if b > a else lo
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
        import torch
        if lane != 0 or not self.split_small or not (self.split_small[0] <= n <= self.split_small[1]):
            return None
        if self._lane_streams is None:
            self._lane_streams = [torch.cuda.Stream() for _ in range(3)]
        return n // 2, self._lane_streams[0]

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
        from .normalize import SPIKE_MODES
        raw_off = np.asarray(raw_off, dtype=np.int64)
        lo = np.asarray(win_lo, dtype=np.int32)
        hi = np.asarray(win_hi, dtype=np.int32)
        lens = np.diff(raw_off)
        lengths = np.maximum(np.minimum(hi.astype(np.int64), lens - 1) - lo + 1, 0).astype(np.int32)
        return self._pipeline(_IngestRaw(self, host_raw, raw_off, lo, hi, lengths, SPIKE_MODES[spike_removal]),
                              lengths, aut, rev, want_seq, chunk_reads, lanes)

    def call_arrays_vbz(self, host_payload, table, read_chunk, raw_off, win_lo, win_hi, aut, rev,
                        spike_removal: str = 'Brute', want_seq: bool = True, chunk_reads: int = 25000,
                        lanes: int = 2) -> Dict[str, np.ndarray]:
        """``call_arrays_raw`` for reads still VBZ-compressed as their fast5 file stores them (``pack_vbz`` makes
        the arguments): only the chunk bodies (after zstd, ~1.25 B per sample instead of 2) cross PCIe, and the
        StreamVByte / zig-zag delta decode (wstr_vbz_decode_batch) writes the int16 reads on the device.  Same
        result dict, plus ``chunk_status`` (WSTR_VBZ_* per chunk; a read with a bad chunk has undefined results)."""
        from .normalize import SPIKE_MODES
        raw_off = np.asarray(raw_off, dtype=np.int64)
        lo = np.asarray(win_lo, dtype=np.int32)
        hi = np.asarray(win_hi, dtype=np.int32)
        lens = np.diff(raw_off)
        lengths = np.maximum(np.minimum(hi.astype(np.int64), lens - 1) - lo + 1, 0).astype(np.int32)
        ingest = _IngestVBZ(self, host_payload, table, np.asarray(read_chunk, dtype=np.int64), raw_off, lo, hi,
                            lengths, SPIKE_MODES[spike_removal])
        return self._pipeline(ingest, lengths, aut, rev, want_seq, chunk_reads, lanes)

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
        out = self._host_results(n, int(seq_off[-1]) if want_seq else 0)
        with torch.cuda.device(self.device):
            comp = torch.cuda.current_stream()
            if self._copy_stream is None:
                self._copy_stream = (torch.cuda.Stream(), torch.cuda.Stream())
            cs_in, cs_out = self._copy_stream
            # device-side signal and result buffers live on the engine and only ever grow, so the
            # chunk loop makes no allocator calls
            ingest.allocate()
            d_sig = ingest.d_sig
            dev = {k: self._device_buffer(k, n, dt) for k, dt in
                   (('len1', torch.int32), ('len2', torch.int32), ('cost1', torch.float64),
                    ('cost2', torch.float64), ('status', torch.int32), ('ties', torch.int32))}
            if want_seq:
                dev['seq1'] = self._device_buffer('seq1', int(seq_off[-1]), torch.uint8)
                dev['seq2'] = self._device_buffer('seq2', int(seq_off[-1]), torch.uint8)
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
            if n_lanes > 1 and self._lane_streams is None:
                self._lane_streams = [torch.cuda.Stream() for _ in range(3)]
            streams = [comp] + (self._lane_streams[:n_lanes - 1] if n_lanes > 1 else [])
            for st in streams[1:]:
                st.wait_stream(comp)
            for ci, (a, b) in enumerate(chunks):
                ev = sent[ci]
                lane = ci % len(streams)
                st = streams[lane]
                lo = int(off[a])
                hi = min(int(off[b - 1] + ((int(lengths[b - 1]) + 1) & ~1) + 2), d_sig.numel())
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
                    ingest.fetch(a, b, out)
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
        res = {k: out[k][:n].numpy().copy() for k in _SCALARS}
        res['ttest_ties'] = res.pop('ties')
        bad = res['status'] != 0
        if bad.any():
            res['len1'][bad] = -1
            res['len2'][bad] = -1
            res['cost1'][bad] = np.nan
            res['cost2'][bad] = np.nan
        if want_seq:
            res['seq1'] = out['seq1'][:int(seq_off[-1])].numpy()
            res['seq2'] = out['seq2'][:int(seq_off[-1])].numpy()
            res['seq_off'] = seq_off[:-1]
        ingest.finish(res, out, n)
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

    def _host_results(self, n: int, seq_bytes: int):
        """Pinned host buffers for the per-read results, grown on demand and reused."""
        import torch
        cur = self._host_out
        if cur is None or cur['len1'].numel() < n or cur['seq1'].numel() < seq_bytes:
            n_cap = max(n, cur['len1'].numel() if cur else 0)
            s_cap = max(seq_bytes, cur['seq1'].numel() if cur else 0, 1)
            pin = torch.cuda.is_available()
            cur = dict(len1=torch.empty(n_cap, dtype=torch.int32, pin_memory=pin),
                       len2=torch.empty(n_cap, dtype=torch.int32, pin_memory=pin),
                       cost1=torch.empty(n_cap, dtype=torch.float64, pin_memory=pin),
                       cost2=torch.empty(n_cap, dtype=torch.float64, pin_memory=pin),
                       status=torch.empty(n_cap, dtype=torch.int32, pin_memory=pin),
                       ties=torch.empty(n_cap, dtype=torch.int32, pin_memory=pin),
                       seq1=torch.empty(s_cap, dtype=torch.uint8, pin_memory=pin),
                       seq2=torch.empty(s_cap, dtype=torch.uint8, pin_memory=pin))
            self._host_out = cur
        return cur

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
        n = len(raws)
        if n == 0:
            return []
        host, raw_off = pack_raw(raws)
        if windows is None:
            d_raw = self._upload_raw(host)
            return self._call_located(d_raw, raw_off, aut_ids, reverse, spike_removal, offset,
                                      lambda idx: [raws[r] for r in idx])
        aut = _single_ids(aut_ids)
        rev = np.asarray(reverse, dtype=np.uint8)
        lo = np.array([w[0] for w in windows], dtype=np.int32)
        hi = np.array([w[1] for w in windows], dtype=np.int32)
        if (lo < 0).any():
            raise ValueError('negative window start')
        res = self.call_arrays_raw(host, raw_off, lo, hi, aut, rev, spike_removal)
        return self._raw_results(res, lambda idx: [raws[r] for r in idx], windows, aut_ids, reverse, spike_removal)

    def call_vbz_batch(self, reads, windows, aut_ids, reverse, spike_removal: str = 'Brute',
                       offset: float = 0.35) -> list:
        """``call_raw_batch`` for reads as their fast5 files store them (fast5.CompressedRead, from
        ``fast5.raw_chunks``): the chunk bodies go to the device, are decoded there (wstr_vbz_decode_batch) and
        called as ``call_raw_batch`` calls raw reads.  A chunk the host decoder would refuse raises that
        Fast5FormatError, naming the file and the read, before any result is returned.  ``windows=None``
        locates the windows first (``locate_arrays_vbz``): the payload crosses PCIe once and the decoded reads
        stay on the device for the call; reads not found come back as ``NotLocated``.  Strand pairs in ``aut_ids``
        as in ``call_raw_batch``."""
        n = len(reads)
        if n == 0:
            return []
        if any(r.n_samples <= 0 for r in reads):
            raise ValueError('empty raw read')
        host, table, read_chunk, raw_off = pack_vbz(reads)
        if windows is None:
            d_raw, chunk_status = self._decode_vbz(host, table, raw_off)
            _raise_bad_chunk(reads, read_chunk, chunk_status.cpu().numpy())
            return self._call_located(d_raw, raw_off, aut_ids, reverse, spike_removal, offset,
                                      lambda idx: [reads[r].decode() for r in idx])
        aut = _single_ids(aut_ids)
        rev = np.asarray(reverse, dtype=np.uint8)
        lo = np.array([w[0] for w in windows], dtype=np.int32)
        hi = np.array([w[1] for w in windows], dtype=np.int32)
        if (lo < 0).any():
            raise ValueError('negative window start')
        res = self.call_arrays_vbz(host, table, read_chunk, raw_off, lo, hi, aut, rev, spike_removal)
        _raise_bad_chunk(reads, read_chunk, res['chunk_status'])
        return self._raw_results(res, lambda idx: [reads[r].decode() for r in idx], windows, aut_ids, reverse,
                                 spike_removal)

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
        raw_off = np.asarray(raw_off, dtype=np.int64)
        return self._locate_device(self._upload_raw(host_raw), raw_off, aut, spike_removal, offset)

    def locate_arrays_vbz(self, host_payload, table, read_chunk, raw_off, aut, spike_removal: str = 'Brute',
                          offset: float = 0.35) -> Dict[str, np.ndarray]:
        """``locate_arrays_raw`` for VBZ-compressed reads (``pack_vbz``): decoded on the device first.  The dict
        also carries ``chunk_status`` (WSTR_VBZ_* per chunk; a read with a bad chunk has undefined results)."""
        raw_off = np.asarray(raw_off, dtype=np.int64)
        d_raw, chunk_status = self._decode_vbz(host_payload, table, raw_off)
        res = self._locate_device(d_raw, raw_off, aut, spike_removal, offset)
        res['chunk_status'] = chunk_status.cpu().numpy()
        return res

    def _upload_raw(self, host_raw):
        import torch
        with torch.cuda.device(self.device):
            d_raw = self._device_buffer('loc_raw16', int(host_raw.numel()), torch.int16)
            d_raw.copy_(host_raw, non_blocking=True)
        return d_raw

    def _decode_vbz(self, host_payload, table, raw_off):
        """Payload -> device -> decoded whole int16 reads (device) and the per-chunk status (device)."""
        import torch
        m = len(table['in_off'])
        with torch.cuda.device(self.device):
            d_pay = self._device_buffer('vbz_payload', int(host_payload.numel()), torch.uint8)
            d_pay.copy_(host_payload, non_blocking=True)
            d_raw = self._device_buffer('loc_raw16', int(raw_off[-1]), torch.int16)
            d_st = torch.zeros(max(m, 1), dtype=torch.int32, device=self.device)
            if m:
                ws = self._device_buffer('vbz_ws0', _lib.vbz_workspace_bytes(m), torch.uint8)
                _lib.vbz_decode_batch(d_pay, table['in_off'], table['in_bytes'], table['n_samples'], table['n_out'],
                                      table['kind'], table['zigzag'], table['out_off'], d_raw, d_st, ws)
        return d_raw, d_st[:m]

    def _locate_device(self, d_raw, raw_off, aut, spike_removal, offset) -> Dict[str, np.ndarray]:
        """Whole-read normalisation of int16 reads on the device, then the window search."""
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
            res = self.locate_packed(d_sig, sig_off, lengths, aut, offset)
            del d_sig
        return res

    def _call_located(self, d_raw, raw_off, aut_ids, reverse, spike_removal, offset, raws_of) -> list:
        """The located-then-called chain on whole int16 reads already on the device: locate, bring the windows
        to the host, normalise the found windows and call them from the same device buffer, each with the
        automaton and orientation of its strand (given, or chosen by the both-strand search)."""
        import torch
        from .normalize import SPIKE_MODES
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
            sub_off = np.zeros(len(found) + 1, dtype=np.int64)
            sub_off[1:] = np.cumsum(np.diff(raw_off)[found])
        else:
            sub_off = raw_off
        lo, hi = loc['lo'][found], loc['hi'][found]
        lengths = (hi - lo + 1).astype(np.int32)
        ingest = _IngestDeviceRaw(self, d_raw, sub_off, lo, hi, lengths, SPIKE_MODES[spike_removal])
        res = self._pipeline(ingest, lengths, aut[found], rev[found], True, 25000, 2)
        windows = list(zip(lo.tolist(), hi.tolist()))
        calls = self._raw_results(res, lambda idx: raws_of([int(found[k]) for k in idx]), windows,
                                  aut[found].tolist(), [bool(x) for x in rev[found]], spike_removal)
        for k, r in enumerate(found):
            out[r] = calls[k]
        return out

    def _raw_results(self, res, raws_of, windows, aut_ids, reverse, spike_removal) -> List[CallerResult]:
        """CallerResults of a ``call_arrays_raw``-style result dict.  Reads the device did not finish, or whose
        t-test decision was within rounding of flipping, are redone as in results_from (the reference's
        exception, or the host's libm for a t-test tie) from their host int16 samples, ``raws_of(indices)``."""
        status, ties = res['status'], res['ttest_ties']
        self.last_ttest_ties = int((ties > 0).sum())
        out: List[Optional[CallerResult]] = []
        redo = []
        so = res['seq_off']
        for r in range(len(status)):
            if status[r] == 0 and ties[r] == 0:
                a = int(so[r])
                out.append(CallerResult(seq=res['seq1'][a:a + res['len1'][r]].tobytes().decode('ascii'),
                                        cost=float(res['cost1'][r]),
                                        resc_seq=res['seq2'][a:a + res['len2'][r]].tobytes().decode('ascii'),
                                        resc_cost=float(res['cost2'][r])))
            else:
                out.append(None)
                redo.append(r)
        if redo:
            from .normalize import normalize_windows
            sigs = normalize_windows(raws_of(redo), [windows[r] for r in redo], spike_removal,
                                     device=str(self.device))
            fixed = self._call_batch_host(sigs, [aut_ids[r] for r in redo], [reverse[r] for r in redo])
            for r, f in zip(redo, fixed):
                out[r] = f
        return out

    def results_from(self, o, signals, aut_ids, reverse) -> List[CallerResult]:
        """Device results -> CallerResult list; reads the device could not finish (status != 0)
        are redone on the host path or raise what the reference raises."""
        status = o['status'].cpu().numpy()
        ties = o['ties'].cpu().numpy() if 'ties' in o else np.zeros_like(status)
        self.last_ttest_ties = int((ties > 0).sum())
        len1, len2 = o['len1'].cpu().numpy(), o['len2'].cpu().numpy()
        cost1, cost2 = o['cost1'].cpu().numpy(), o['cost2'].cpu().numpy()
        seq1, seq2 = o['seq1'].cpu().numpy(), o['seq2'].cpu().numpy()
        off = o['seq_off']
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
            fixed = self._call_batch_host([signals[r] for r in redo], [aut_ids[r] for r in redo],
                                          [reverse[r] for r in redo])
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


def _raise_bad_chunk(reads, read_chunk, chunk_status) -> None:
    """The Fast5FormatError of the first chunk the device decoder refused, naming the file and the read."""
    from .fast5 import Fast5FormatError
    bad = np.flatnonzero(chunk_status)
    if len(bad):
        c = int(bad[0])
        r = int(np.searchsorted(read_chunk, c, side='right')) - 1
        msg = _lib.VBZ_STATUS_MESSAGES.get(int(chunk_status[c]), 'VBZ: corrupt chunk')
        raise Fast5FormatError(f'{reads[r].path}: read {reads[r].read_name}: {msg} '
                               f'(chunk at sample {reads[r].chunks[c - int(read_chunk[r])].start})')


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
