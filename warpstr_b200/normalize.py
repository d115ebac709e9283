"""Per-read normalisation on the GPU: spike removal + MAD normalisation + window slice.

Mirrors the numerics of the reference's ``Fast5.get_data_processed`` / ``remove_spikes`` /
``normalize_signal_mad`` (schemas/fast5.py:45-57, 68-77, 90-114) for raw int16 reads that are
already in memory (``fast5.py`` reads them from the fast5 container).  All reads of a
batch are processed by one launch of ``wstr_normalize_batch``.
"""
from typing import Optional, Sequence, Tuple

import numpy as np

from . import _lib
from .pore_model import mad_normalize_float

SPIKE_MODES = {'None': 0, 'Brute': 1, 'median3': 3, 'median5': 5}


def normalize_windows(raws: Sequence[np.ndarray], windows: Sequence[Tuple[int, int]],
                      spike_removal: str = 'Brute', device: str = 'cuda',
                      return_shift_scale: bool = False):
    """For every raw int16 read return the float64 normalised samples of
    ``[l_start_raw, r_end_raw]`` (inclusive, clipped at the read's end like a numpy slice)."""
    import torch
    from .caller import _window_bounds, pack_raw
    if spike_removal not in SPIKE_MODES:
        raise AssertionError('spike_removal must be None, median3, median5 or Brute')
    n = len(raws)
    if n == 0:
        return ([], np.zeros((0, 2))) if return_shift_scale else []
    dev = torch.device(device)
    host, raw_off = pack_raw(raws)
    lo, hi, out_len = _window_bounds(raw_off, [w[0] for w in windows], [w[1] for w in windows])
    out_off = np.zeros(n, dtype=np.int64)
    out_off[1:] = np.cumsum(out_len[:-1])
    with torch.cuda.device(dev):
        d_raw = host.to(dev, non_blocking=True)
        d_out = torch.empty(max(int(out_len.sum()), 1), dtype=torch.float64, device=dev)
        d_ss = torch.empty(2 * n, dtype=torch.float64, device=dev)
        ws = torch.empty(_lib.normalize_workspace_bytes(n), dtype=torch.uint8, device=dev)
        _lib.normalize_batch(d_raw, raw_off, lo, hi, SPIKE_MODES[spike_removal], d_out, out_off, d_ss, ws)
        out = d_out.cpu().numpy()
        ss = d_ss.cpu().numpy().reshape(n, 2)
    res = [out[o:o + ln].copy() for o, ln in zip(out_off, out_len)]
    return (res, ss) if return_shift_scale else res


def normalize_signal_mad(data) -> np.ndarray:
    """Reference-named entry point (fast5.py:104-114).  int16 input runs on the GPU;
    float input (the 4096-row pore table) is a one-off host computation."""
    arr = np.asarray(data)
    if arr.dtype == np.int16:
        return normalize_windows([arr], [(0, len(arr) - 1)], 'None')[0]
    return mad_normalize_float(arr)


def get_data_processed(raw: np.ndarray, position: Optional[Tuple[int, int]] = None,
                       spike_removal: str = 'Brute') -> np.ndarray:
    """Fast5.get_data_processed for one in-memory read (fast5.py:45-57)."""
    raw = np.asarray(raw, dtype=np.int16)
    win = position if position is not None else (0, len(raw) - 1)
    return normalize_windows([raw], [win], spike_removal)[0]
