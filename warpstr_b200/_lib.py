"""ctypes binding of libwarpstr_b200.so (include/warpstr_b200.h).

PyTorch is used for device buffers and streams only; every compute call goes
through the C ABI with raw device pointers.  There is no CPU fallback: if the
shared library is missing, or a call fails, this module raises.
"""
import ctypes
import os
from typing import List, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('WSTR_LIB') or os.path.join(_HERE, 'libwarpstr_b200.so')

_lib = None


class WarpstrError(RuntimeError):
    pass


c_i32p = ctypes.POINTER(ctypes.c_int32)
c_i64p = ctypes.POINTER(ctypes.c_int64)
c_f64p = ctypes.POINTER(ctypes.c_double)
c_u8p = ctypes.POINTER(ctypes.c_uint8)
c_vp = ctypes.c_void_p

class CallParams(ctypes.Structure):
    _fields_ = [('min_values_per_state', ctypes.c_int32), ('states_in_segment', ctypes.c_int32),
                ('threshold', ctypes.c_double), ('max_std', ctypes.c_double),
                ('method', ctypes.c_int32), ('reps_as_one', ctypes.c_int32),
                ('ttest_guard_ulps', ctypes.c_int64)]


class CallOutputs(ctypes.Structure):
    _fields_ = [('d_len1', ctypes.c_void_p), ('d_len2', ctypes.c_void_p), ('d_cost1', ctypes.c_void_p),
                ('d_cost2', ctypes.c_void_p), ('d_status', ctypes.c_void_p), ('d_seq1', ctypes.c_void_p),
                ('d_seq2', ctypes.c_void_p), ('seq_off', ctypes.POINTER(ctypes.c_int64)),
                ('d_trace1', ctypes.c_void_p), ('d_trace2', ctypes.c_void_p), ('d_rescaled', ctypes.c_void_p),
                ('d_ttest_ties', ctypes.c_void_p)]


_SIGNATURES = {
    'wstr_version': (ctypes.c_int, []),
    'wstr_error_string': (ctypes.c_char_p, [ctypes.c_int]),
    'wstr_last_cuda_error': (ctypes.c_char_p, []),
    'wstr_pore_lookup': (ctypes.c_int, [c_vp, ctypes.c_int64, c_vp, ctypes.c_int32, c_vp, c_vp, c_vp]),
    'wstr_normalize_workspace_bytes': (ctypes.c_int64, [ctypes.c_int32]),
    'wstr_normalize_batch': (ctypes.c_int, [c_vp, c_i64p, c_i32p, c_i32p, ctypes.c_int32, ctypes.c_int32,
                                            c_vp, c_i64p, c_vp, c_vp, ctypes.c_int64, c_vp]),
    'wstr_dequantize_workspace_bytes': (ctypes.c_int64, [ctypes.c_int32]),
    'wstr_dequantize_batch': (ctypes.c_int, [c_vp, c_i64p, c_i32p, c_vp, ctypes.c_int32, c_vp, c_i64p, c_vp,
                                             ctypes.c_int64, c_vp]),
    'wstr_vbz_workspace_bytes': (ctypes.c_int64, [ctypes.c_int32]),
    'wstr_vbz_decode_batch': (ctypes.c_int, [c_vp, c_i64p, c_i64p, c_i32p, c_i32p, c_i32p, c_i32p, c_i64p,
                                             ctypes.c_int32, c_vp, c_vp, c_vp, ctypes.c_int64, c_vp]),
    'wstr_zstd_workspace_bytes': (ctypes.c_int64, [ctypes.c_int32]),
    'wstr_zstd_decode_batch': (ctypes.c_int, [c_vp, c_i64p, c_i64p, c_i64p, c_i64p, ctypes.c_int32, c_vp, c_vp, c_vp,
                                              ctypes.c_int64, c_vp]),
    'wstr_automaton_create': (ctypes.c_int, [c_f64p, c_i32p, c_i32p, c_i32p, c_u8p, c_u8p, ctypes.c_int32,
                                             ctypes.c_int32, ctypes.c_int32, ctypes.c_int32,
                                             ctypes.POINTER(c_vp)]),
    'wstr_automaton_destroy': (ctypes.c_int, [c_vp]),
    'wstr_set_generic_only': (ctypes.c_int, [ctypes.c_int32]),
    'wstr_automaton_plan': (ctypes.c_int, [c_i32p, c_i32p, ctypes.c_int32, ctypes.c_int32, c_i32p, c_i32p,
                                           ctypes.c_int32]),
    'wstr_automaton_info': (ctypes.c_int, [c_vp, c_i32p, ctypes.c_int32]),
    'wstr_automaton_layout': (ctypes.c_int, [c_vp, c_i32p, ctypes.c_int32]),
    'wstr_warp_workspace_bytes': (ctypes.c_int64, [ctypes.POINTER(c_vp), ctypes.c_int32, c_i32p, c_i32p,
                                                   ctypes.c_int32]),
    'wstr_warp_batch': (ctypes.c_int, [ctypes.POINTER(c_vp), ctypes.c_int32, c_i32p, c_vp, c_i64p, c_i32p,
                                       c_vp, c_i64p, ctypes.c_int32, c_vp, ctypes.c_int64, c_vp, c_vp, c_vp,
                                       c_vp]),
    'wstr_measure_fp64_add_rate': (ctypes.c_int, [c_f64p, c_vp]),
    'wstr_call_workspace_bytes': (ctypes.c_int64, [ctypes.POINTER(c_vp), ctypes.c_int32, c_i32p, c_i32p,
                                                   ctypes.c_int32]),
    'wstr_call_workspace_min_bytes': (ctypes.c_int64, [ctypes.POINTER(c_vp), ctypes.c_int32, c_i32p, c_i32p,
                                                       ctypes.c_int32]),
    'wstr_call_batch': (ctypes.c_int, [ctypes.POINTER(c_vp), ctypes.c_int32, c_i32p, c_u8p, c_vp, c_i64p, c_i32p,
                                       ctypes.c_int32, ctypes.POINTER(CallParams), c_vp, ctypes.c_int64,
                                       ctypes.POINTER(CallOutputs), c_vp]),
    'wstr_locate_workspace_bytes': (ctypes.c_int64, [ctypes.POINTER(c_vp), ctypes.c_int32, ctypes.c_int32]),
    'wstr_locate_batch': (ctypes.c_int, [ctypes.POINTER(c_vp), ctypes.c_int32, c_i32p, c_vp, c_i64p, c_i32p,
                                         ctypes.c_int32, ctypes.c_double, c_vp, c_vp, c_vp, c_vp, c_vp, ctypes.c_int64,
                                         c_vp]),
    'wstr_assign_workspace_bytes': (ctypes.c_int64, [ctypes.POINTER(c_vp), ctypes.c_int32, ctypes.c_int32]),
    'wstr_assign_batch': (ctypes.c_int, [ctypes.POINTER(c_vp), ctypes.c_int32, c_vp, c_i64p, c_i32p, ctypes.c_int32,
                                         ctypes.c_double, c_vp, c_vp, c_vp, c_vp, ctypes.c_int64, c_vp]),
    'wstr_profile_enable': (ctypes.c_int, [ctypes.c_int32]),
    'wstr_profile_read': (ctypes.c_int, [c_f64p, c_i32p, ctypes.c_int32]),
}


def lib():
    """The loaded shared library; raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise WarpstrError(
                f'{LIB_PATH} not found: build it with `python -c "import __graft_entry__ as g; g.build()"` '
                '(there is no CPU fallback)')
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def exported_symbols() -> List[str]:
    return list(_SIGNATURES)


def check(rc: int, what: str = '') -> None:
    if rc == 0:
        return
    L = lib()
    msg = L.wstr_error_string(int(rc)).decode()
    cuda = L.wstr_last_cuda_error().decode()
    raise WarpstrError(f'{what or "warpstr_b200"} failed: {msg}' + (f' [{cuda}]' if cuda and rc == -2 else ''))


def _np(a, dtype):
    return np.ascontiguousarray(a, dtype=dtype)


def _ptr(a, ty):
    return a.ctypes.data_as(ty)


def _stream_ptr(stream=None):
    import torch
    s = stream if stream is not None else torch.cuda.current_stream()
    return ctypes.c_void_p(s.cuda_stream)


def _dptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


# ---------------------------------------------------------------------------------------
class DeviceAutomaton:
    """Owns a ``wstr_automaton`` handle (device-resident kernel tables of one strand)."""

    def __init__(self, values, seq_idx, in_ptr, in_idx, rep_mask, last_base, endstate: int,
                 flank_length: int, min_values_per_state: int = 4):
        import torch
        if not torch.cuda.is_available():
            raise WarpstrError('warpstr_b200 needs a CUDA device (there is no CPU fallback)')
        values = _np(values, np.float64)
        seq_idx = _np(seq_idx, np.int32)
        in_ptr = _np(in_ptr, np.int32)
        in_idx = _np(in_idx, np.int32)
        rep_mask = _np(rep_mask, np.uint8)
        last_base = _np(last_base, np.uint8)
        self.n_states = int(values.shape[0])
        self.flank_length = int(flank_length)
        self.min_values_per_state = int(min_values_per_state)
        self.handle = c_vp()
        rc = lib().wstr_automaton_create(
            _ptr(values, c_f64p), _ptr(seq_idx, c_i32p), _ptr(in_ptr, c_i32p), _ptr(in_idx, c_i32p),
            _ptr(rep_mask, c_u8p), _ptr(last_base, c_u8p), self.n_states, int(endstate), int(flank_length),
            int(min_values_per_state), ctypes.byref(self.handle))
        check(rc, 'wstr_automaton_create')

    @classmethod
    def from_automaton(cls, sta, flank_length: int, min_values_per_state: int = 4):
        return cls(sta.values, sta.seq_idx, sta.in_ptr, sta.in_idx, sta.rep_mask, sta.last_base,
                   sta.endstate, flank_length, min_values_per_state)

    def info(self) -> dict:
        buf = np.zeros(9, dtype=np.int32)
        check(lib().wstr_automaton_info(self.handle, _ptr(buf, c_i32p), 9), 'wstr_automaton_info')
        keys = ('states_per_lane', 'dir_bits_per_row', 'chain_slots', 'generic_slots', 'n_states', 'n_edges',
                'generic_states', 'band_closed', 'unrolled_in_degree')
        return dict(zip(keys, (int(x) for x in buf)))

    def layout(self) -> np.ndarray:
        n = 32 * self.info()['states_per_lane']
        buf = np.zeros(n, dtype=np.int32)
        check(lib().wstr_automaton_layout(self.handle, _ptr(buf, c_i32p), n), 'wstr_automaton_layout')
        return buf

    def close(self):
        if getattr(self, 'handle', None) and self.handle.value:
            lib().wstr_automaton_destroy(self.handle)
            self.handle = c_vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def automaton_plan(in_ptr, in_idx, n_states: int, min_values_per_state: int = 4):
    """Host-only dry run of the kernel layout: (info dict, state_of_pos)."""
    ip = _np(in_ptr, np.int32)
    ii = _np(in_idx, np.int32)
    info = np.zeros(5, dtype=np.int32)
    sop = np.full(32 * 16, -1, dtype=np.int32)
    check(lib().wstr_automaton_plan(_ptr(ip, c_i32p), _ptr(ii, c_i32p), int(n_states), int(min_values_per_state),
                                    _ptr(info, c_i32p), _ptr(sop, c_i32p), int(sop.shape[0])), 'wstr_automaton_plan')
    keys = ('chain_slots', 'generic_slots', 'unrolled_in_degree', 'chain_lanes', 'generic_states')
    d = dict(zip(keys, (int(x) for x in info)))
    return d, sop[:32 * (d['chain_slots'] + d['generic_slots'])]


def set_generic_only(on: bool) -> None:
    """Testing aid: automata created while this is on use the catch-all kernel."""
    check(lib().wstr_set_generic_only(1 if on else 0), 'wstr_set_generic_only')


def _handles(automata: Sequence[DeviceAutomaton]):
    arr = (c_vp * len(automata))(*[a.handle.value for a in automata])
    return arr


def warp_workspace_bytes(automata: Sequence[DeviceAutomaton], read_automaton: np.ndarray,
                         lengths: np.ndarray) -> int:
    ra = _np(read_automaton, np.int32)
    ln = _np(lengths, np.int32)
    n = lib().wstr_warp_workspace_bytes(_handles(automata), len(automata), _ptr(ra, c_i32p), _ptr(ln, c_i32p),
                                        int(ln.shape[0]))
    if n < 0:
        check(int(n), 'wstr_warp_workspace_bytes')
    return int(n)


def warp_batch(automata: Sequence[DeviceAutomaton], read_automaton, d_signal, sig_off, lengths,
               d_maskbits, mask_off, d_workspace, d_trace, d_end_cost, d_status, stream=None) -> None:
    ra = _np(read_automaton, np.int32)
    so = _np(sig_off, np.int64)
    ln = _np(lengths, np.int32)
    mo = _np(mask_off, np.int64) if mask_off is not None else None
    rc = lib().wstr_warp_batch(
        _handles(automata), len(automata), _ptr(ra, c_i32p), _dptr(d_signal), _ptr(so, c_i64p), _ptr(ln, c_i32p),
        _dptr(d_maskbits), _ptr(mo, c_i64p) if mo is not None else None, int(ln.shape[0]),
        _dptr(d_workspace), int(d_workspace.numel() * d_workspace.element_size()),
        _dptr(d_trace), _dptr(d_end_cost), _dptr(d_status), _stream_ptr(stream))
    check(rc, 'wstr_warp_batch')


def pore_lookup(d_seq, d_table, k: int, d_out, d_bad, stream=None) -> None:
    rc = lib().wstr_pore_lookup(_dptr(d_seq), int(d_seq.numel()), _dptr(d_table), int(k), _dptr(d_out),
                                _dptr(d_bad), _stream_ptr(stream))
    check(rc, 'wstr_pore_lookup')


def normalize_workspace_bytes(n_reads: int) -> int:
    n = lib().wstr_normalize_workspace_bytes(int(n_reads))
    if n < 0:
        check(int(n), 'wstr_normalize_workspace_bytes')
    return int(n)


def normalize_batch(d_raw, raw_off, win_lo, win_hi, spike_mode: int, d_out, out_off, d_shift_scale,
                    d_workspace, stream=None) -> None:
    ro = _np(raw_off, np.int64)
    lo = _np(win_lo, np.int32)
    hi = _np(win_hi, np.int32)
    oo = _np(out_off, np.int64)
    rc = lib().wstr_normalize_batch(
        _dptr(d_raw), _ptr(ro, c_i64p), _ptr(lo, c_i32p), _ptr(hi, c_i32p), int(lo.shape[0]), int(spike_mode),
        _dptr(d_out), _ptr(oo, c_i64p), _dptr(d_shift_scale), _dptr(d_workspace),
        int(d_workspace.numel() * d_workspace.element_size()), _stream_ptr(stream))
    check(rc, 'wstr_normalize_batch')


def dequantize_batch(d_raw, raw_off, lengths, d_shift_scale, d_out, out_off, d_workspace, stream=None) -> None:
    ro = _np(raw_off, np.int64)
    ln = _np(lengths, np.int32)
    oo = _np(out_off, np.int64)
    rc = lib().wstr_dequantize_batch(_dptr(d_raw), _ptr(ro, c_i64p), _ptr(ln, c_i32p), _dptr(d_shift_scale),
                                     int(ln.shape[0]), _dptr(d_out), _ptr(oo, c_i64p), _dptr(d_workspace),
                                     int(d_workspace.numel() * d_workspace.element_size()), _stream_ptr(stream))
    check(rc, 'wstr_dequantize_batch')


VBZ_KIND_V0, VBZ_KIND_V1, VBZ_KIND_RAW = 0, 1, 2
# d_status of wstr_vbz_decode_batch -> the message fast5.vbz_decompress raises for the same chunk
VBZ_STATUS_MESSAGES = {
    1: 'VBZ: truncated StreamVByte control block',
    2: 'VBZ: truncated StreamVByte data block',
    3: 'VBZ v1: data block length does not match the keys',
}


def vbz_workspace_bytes(n_chunks: int) -> int:
    n = lib().wstr_vbz_workspace_bytes(int(n_chunks))
    if n < 0:
        check(int(n), 'wstr_vbz_workspace_bytes')
    return int(n)


def vbz_decode_batch(d_payload, in_off, in_bytes, n_samples, n_out, kind, zigzag, out_off, d_raw, d_status,
                     d_workspace, stream=None) -> None:
    io = _np(in_off, np.int64)
    ib = _np(in_bytes, np.int64)
    ns = _np(n_samples, np.int32)
    no = _np(n_out, np.int32)
    kd = _np(kind, np.int32)
    zz = _np(zigzag, np.int32)
    oo = _np(out_off, np.int64)
    rc = lib().wstr_vbz_decode_batch(
        _dptr(d_payload), _ptr(io, c_i64p), _ptr(ib, c_i64p), _ptr(ns, c_i32p), _ptr(no, c_i32p), _ptr(kd, c_i32p),
        _ptr(zz, c_i32p), _ptr(oo, c_i64p), int(io.shape[0]), _dptr(d_raw), _dptr(d_status), _dptr(d_workspace),
        int(d_workspace.numel() * d_workspace.element_size()), _stream_ptr(stream))
    check(rc, 'wstr_vbz_decode_batch')


def zstd_workspace_bytes(n_frames: int) -> int:
    n = lib().wstr_zstd_workspace_bytes(int(n_frames))
    if n < 0:
        check(int(n), 'wstr_zstd_workspace_bytes')
    return int(n)


def zstd_decode_batch(d_in, in_off, in_bytes, out_off, out_bytes, d_out, d_status, d_workspace, stream=None) -> None:
    io = _np(in_off, np.int64)
    ib = _np(in_bytes, np.int64)
    oo = _np(out_off, np.int64)
    ob = _np(out_bytes, np.int64)
    rc = lib().wstr_zstd_decode_batch(
        _dptr(d_in), _ptr(io, c_i64p), _ptr(ib, c_i64p), _ptr(oo, c_i64p), _ptr(ob, c_i64p), int(io.shape[0]),
        _dptr(d_out), _dptr(d_status), _dptr(d_workspace), int(d_workspace.numel() * d_workspace.element_size()),
        _stream_ptr(stream))
    check(rc, 'wstr_zstd_decode_batch')


def measure_fp64_add_rate(stream=None) -> float:
    out = ctypes.c_double(0.0)
    check(lib().wstr_measure_fp64_add_rate(ctypes.byref(out), _stream_ptr(stream)), 'wstr_measure_fp64_add_rate')
    return float(out.value)


def call_workspace_bytes(automata: Sequence[DeviceAutomaton], read_automaton, lengths) -> int:
    ra = _np(read_automaton, np.int32)
    ln = _np(lengths, np.int32)
    n = lib().wstr_call_workspace_bytes(_handles(automata), len(automata), _ptr(ra, c_i32p), _ptr(ln, c_i32p),
                                        int(ln.shape[0]))
    if n < 0:
        check(int(n), 'wstr_call_workspace_bytes')
    return int(n)


def call_workspace_min_bytes(automata: Sequence[DeviceAutomaton], read_automaton, lengths) -> int:
    ra = _np(read_automaton, np.int32)
    ln = _np(lengths, np.int32)
    n = lib().wstr_call_workspace_min_bytes(_handles(automata), len(automata), _ptr(ra, c_i32p), _ptr(ln, c_i32p),
                                            int(ln.shape[0]))
    if n < 0:
        check(int(n), 'wstr_call_workspace_min_bytes')
    return int(n)


def call_batch(automata: Sequence[DeviceAutomaton], read_automaton, read_reverse, d_signal, sig_off, lengths,
               params: CallParams, d_workspace, d_len1, d_len2, d_cost1, d_cost2, d_status, d_seq1=None,
               d_seq2=None, seq_off=None, d_trace1=None, d_trace2=None, d_rescaled=None, stream=None,
               d_ttest_ties=None) -> None:
    ra = _np(read_automaton, np.int32)
    rv = _np(read_reverse, np.uint8)
    so = _np(sig_off, np.int64)
    ln = _np(lengths, np.int32)
    qo = _np(seq_off, np.int64) if seq_off is not None else None
    out = CallOutputs(_dptr(d_len1), _dptr(d_len2), _dptr(d_cost1), _dptr(d_cost2), _dptr(d_status),
                      _dptr(d_seq1), _dptr(d_seq2), _ptr(qo, c_i64p) if qo is not None else None,
                      _dptr(d_trace1), _dptr(d_trace2), _dptr(d_rescaled), _dptr(d_ttest_ties))
    rc = lib().wstr_call_batch(
        _handles(automata), len(automata), _ptr(ra, c_i32p), _ptr(rv, c_u8p), _dptr(d_signal), _ptr(so, c_i64p),
        _ptr(ln, c_i32p), int(ln.shape[0]), ctypes.byref(params), _dptr(d_workspace),
        int(d_workspace.numel() * d_workspace.element_size()), ctypes.byref(out), _stream_ptr(stream))
    check(rc, 'wstr_call_batch')


LOCATE_FOUND, LOCATE_NOT_FOUND, LOCATE_NO_PATH = 0, 1, 2     # d_status of wstr_locate_batch
LOCATE_MAX_SAMPLES = 2**31 - 4096


def locate_workspace_bytes(automata: Sequence[DeviceAutomaton], n_reads: int) -> int:
    n = lib().wstr_locate_workspace_bytes(_handles(automata), len(automata), int(n_reads))
    if n < 0:
        check(int(n), 'wstr_locate_workspace_bytes')
    return int(n)


def locate_batch(automata: Sequence[DeviceAutomaton], read_automaton, d_signal, sig_off, lengths, offset: float,
                 d_lo, d_hi, d_score, d_status, d_workspace, stream=None) -> None:
    ra = _np(read_automaton, np.int32)
    so = _np(sig_off, np.int64)
    ln = _np(lengths, np.int32)
    rc = lib().wstr_locate_batch(
        _handles(automata), len(automata), _ptr(ra, c_i32p), _dptr(d_signal), _ptr(so, c_i64p), _ptr(ln, c_i32p),
        int(ln.shape[0]), float(offset), _dptr(d_lo), _dptr(d_hi), _dptr(d_score), _dptr(d_status),
        _dptr(d_workspace), int(d_workspace.numel() * d_workspace.element_size()), _stream_ptr(stream))
    check(rc, 'wstr_locate_batch')


# wstr_assign_hit: one (read, locus) whose flanks were found on a strand
ASSIGN_HIT = np.dtype([('read', np.int32), ('locus', np.int32), ('strand', np.int32), ('pad_', np.int32),
                       ('left_lo', np.int32), ('left_hi', np.int32), ('right_lo', np.int32), ('right_hi', np.int32),
                       ('left_score', np.float64), ('right_score', np.float64)])


def assign_workspace_bytes(automata: Sequence[DeviceAutomaton], n_reads: int) -> int:
    n = lib().wstr_assign_workspace_bytes(_handles(automata), len(automata), int(n_reads))
    if n < 0:
        check(int(n), 'wstr_assign_workspace_bytes')
    return int(n)


def assign_batch(automata: Sequence[DeviceAutomaton], d_signal, sig_off, lengths, offset: float, d_table, d_hits,
                 d_n_hits, d_workspace, stream=None) -> None:
    """wstr_assign_batch.  ``d_table``: None, or a uint8 tensor of 20 * n_reads * len(automata) bytes (the header's
    struct of arrays, see ``split_table``); ``d_hits``: a uint8 tensor with room for n_reads * len(automata) / 4
    ASSIGN_HIT records; ``d_n_hits``: one int32."""
    so = _np(sig_off, np.int64)
    ln = _np(lengths, np.int32)
    rc = lib().wstr_assign_batch(
        _handles(automata), len(automata), _dptr(d_signal), _ptr(so, c_i64p), _ptr(ln, c_i32p), int(ln.shape[0]),
        float(offset), _dptr(d_table), _dptr(d_hits), _dptr(d_n_hits), _dptr(d_workspace),
        int(d_workspace.numel() * d_workspace.element_size()), _stream_ptr(stream))
    check(rc, 'wstr_assign_batch')


def split_table(buf: np.ndarray, n_reads: int, n_automata: int):
    """The bytes of wstr_assign_batch's d_table -> (lo, hi, score, status), each [n_reads, n_automata]."""
    m = n_reads * n_automata
    buf = np.ascontiguousarray(buf, dtype=np.uint8)
    score = buf[:8 * m].view(np.float64)
    lo, hi, status = (buf[8 * m + 4 * m * k:8 * m + 4 * m * (k + 1)].view(np.int32) for k in range(3))
    return tuple(a.reshape(n_reads, n_automata) for a in (lo, hi, score, status))


PROFILE_CATEGORIES =('dp_fill_traceback', 'midstage', 'normalize', 'pore_lookup', 'plan_upload')


def profile_enable(on: bool = True) -> None:
    check(lib().wstr_profile_enable(1 if on else 0), 'wstr_profile_enable')


def profile_read() -> dict:
    n = len(PROFILE_CATEGORIES)
    ms = np.zeros(n, dtype=np.float64)
    cnt = np.zeros(n, dtype=np.int32)
    check(lib().wstr_profile_read(_ptr(ms, c_f64p), _ptr(cnt, c_i32p), n), 'wstr_profile_read')
    return {name: {'ms': float(ms[i]), 'launches': int(cnt[i])} for i, name in enumerate(PROFILE_CATEGORIES)}
