"""Measures the STR window search in whole reads (wstr_locate_batch, DESIGN.md section 4.5).

    python scripts/bench_locate.py --out profiles/r04_locate.json

1. Locate rate (reads/s, DP cells/s with cells = N x S per read) of CallerEngine.locate_packed on device-resident
   whole normalised reads of ~150 000 samples (HD locus), for 10 and 2 000 reads, against the FP64 add rate
   measured in the same run (wstr_measure_fp64_add_rate).  A cell costs at least mv + 1 + in-degree FP64 adds.
   Strand mode, on the same reads: the single-strand search with the true strands against the both-strand search
   (every read a (template, reverse) pair, two entries per read; its cells count both strands), alternated.
2. Files to overview.csv: main_wrapper on multi-read VBZ fast5 files of a caller-only overview, with every
   window given, with the window columns left empty (located first) and with the window and ``reverse``
   columns left empty (located on both strands), on the same files.
Card name and power limit are read in the same run and written beside the numbers.
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))


def gpu_info():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else 'unknown'
    except Exception as e:   # noqa: BLE001
        return f'unknown ({e})'


def whole_reads(locus, n, samples, seed):
    """Synthetic whole reads: make_reads windows in squiggled random sequence, ~``samples`` each."""
    from warpstr_b200 import synth
    pm = synth.get_pore_model()
    rng = np.random.default_rng(seed)
    reads = synth.make_reads(locus, n, seed=seed)
    sigs, wins = [], []
    for r in reads:
        pad = max(samples - len(r.signal), 2)
        a = int(rng.integers(pad // 4, 3 * pad // 4))
        fill = synth.squiggle(rng, synth.random_flank(rng, pad // 9 + 8), pm)[:pad]
        sigs.append(np.concatenate((fill[:a], r.signal, fill[a:])))
        wins.append((a, a + len(r.signal) - 1))
    return sigs, wins, [r.reverse for r in reads]


def bench_locate(n, samples, reps):
    import torch
    from warpstr_b200 import synth
    from warpstr_b200.automata import StateAutomata
    from warpstr_b200.caller import CallerEngine, pack_signals
    locus = synth.make_locus('HD', seed=3)
    eng = CallerEngine()
    stas = [StateAutomata(locus.template_regex), StateAutomata(locus.reverse_regex)]
    ids = [eng.add_automaton(s, locus.flank_length) for s in stas]
    sigs, wins, rev = whole_reads(locus, n, samples, seed=n)
    host, off, lengths = pack_signals(sigs)
    d_sig = host.to(eng.device)
    aut = [ids[int(r)] for r in rev]
    pairs = [tuple(ids)] * n
    res = eng.locate_packed(d_sig, off, lengths, aut)          # warm-up, also the accuracy figure below
    both = eng.locate_packed(d_sig, off, lengths, pairs)
    torch.cuda.synchronize()
    t, t2 = [], []
    for _ in range(reps):                                      # single and both strands alternated
        t0 = time.perf_counter()
        eng.locate_packed(d_sig, off, lengths, aut)            # ends in a device-to-host copy: synchronised
        t.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        eng.locate_packed(d_sig, off, lengths, pairs)
        t2.append(time.perf_counter() - t0)
    sec, sec2 = float(np.median(t)), float(np.median(t2))
    S = np.array([stas[int(r)].n_states for r in rev], dtype=np.float64)
    cells = float((lengths.astype(np.float64) * S).sum())
    cells2 = float(lengths.astype(np.float64).sum()) * float(stas[0].n_states + stas[1].n_states)
    deg = stas[0].n_edges / stas[0].n_states
    w = np.array(wins)
    err = np.maximum(np.abs(res['lo'] - w[:, 0]), np.abs(res['hi'] - w[:, 1]))
    truth = np.array(rev, dtype=np.int8)
    gap = np.abs(both['strand_score'][:, 0] - both['strand_score'][:, 1])
    return dict(reads=n, samples_per_read=int(np.mean(lengths)), states=int(S.mean()), seconds_median=sec,
                seconds_all=t, reads_per_s=n / sec, cells_per_s=cells / sec,
                fp64_adds_per_cell_min=float(eng.cc.min_values_per_state + 1 + deg),
                found=int((res['status'] == 0).sum()), end_error_max=int(err.max()),
                end_error_p99=float(np.percentile(err, 99)),
                both_strands=dict(seconds_median=sec2, seconds_all=t2, reads_per_s=n / sec2, cells_per_s=cells2 / sec2,
                                  time_over_single_strand=sec2 / sec, right_strand=int((both['strand'] == truth).sum()),
                                  same_window_as_single=int(((both['lo'] == res['lo']) & (both['hi'] == res['hi'])).sum()),
                                  score_gap_min=float(gap.min())))


def bench_files(n_reads, samples, reps):
    """files -> overview.csv with windows given vs located vs located on both strands, same fast5 files."""
    import warnings
    import _h5write as hw
    from warpstr_b200 import caller_only, synth
    from warpstr_b200.wrapper import Locus, flanks_from_template, main_wrapper
    locus = synth.make_locus('HD', seed=5)
    sigs, wins, rev = whole_reads(locus, n_reads, samples, seed=77)
    tmp = tempfile.mkdtemp(prefix='bench_locate_')
    try:
        per_file = [dict() for _ in range(4)]
        rows = []
        for i, (s, (a, b)) in enumerate(zip(sigs, wins)):
            raw = np.rint((90.8717 + 9.8354 * s) * 5.85).astype(np.int16)
            per_file[i % 4][f'{i:05d}-read'] = raw
            rows.append((i % 4, f'{i:05d}-read', rev[i], a, b))
        paths = []
        for k, d in enumerate(per_file):
            p = os.path.join(tmp, f'run{k}.fast5')
            hw.write_multi(p, d, 'vbz0', chunk=4000)
            paths.append(p)
        out = {}
        for mode in ('given', 'located', 'detected'):
            csv_path = os.path.join(tmp, f'{mode}.csv')
            with open(csv_path, 'w') as fh:
                fh.write('fast5_path,locus,read_name,reverse,l_start_raw,r_end_raw\n')
                for k, rid, rv, a, b in rows:
                    win = f'{a},{b}' if mode == 'given' else ','
                    fh.write(f'{paths[k]},LOC,{rid},{rv if mode != "detected" else ""},{win}\n')
            times = []
            for rep in range(reps + 1):
                o = os.path.join(tmp, f'out_{mode}')
                shutil.rmtree(o, ignore_errors=True)
                caller_only.prepare(o, csv_path)
                loc = Locus(name='LOC', sequence=locus.sequence, flank_length=locus.flank_length,
                            path=os.path.join(o, 'LOC'))
                t0 = time.perf_counter()
                with warnings.catch_warnings():
                    warnings.simplefilter('ignore')
                    main_wrapper(loc, flanks=flanks_from_template(locus.left, locus.right))
                if rep:                                   # the first run warms up
                    times.append(time.perf_counter() - t0)
            out[mode] = dict(seconds_median=float(np.median(times)), seconds_all=times)
        out['located_over_given'] = out['located']['seconds_median'] / out['given']['seconds_median']
        out['detected_over_given'] = out['detected']['seconds_median'] / out['given']['seconds_median']
        out['reads'] = n_reads
        out['samples_per_read'] = samples
        return out
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    ap.add_argument('--samples', type=int, default=150_000)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--file-reads', type=int, default=1000)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('bench_locate.py measures the GPU: no CUDA device')
    from warpstr_b200 import _lib
    res = dict(gpu=gpu_info())
    res['fp64_add_rate_tera_per_s'] = _lib.measure_fp64_add_rate()
    res['locate'] = [bench_locate(n, args.samples, args.reps) for n in (10, 2000)]
    for r in res['locate']:
        r['cells_per_fp64_add_rate'] = r['cells_per_s'] / (res['fp64_add_rate_tera_per_s'] * 1e12)
    res['files_to_overview'] = bench_files(args.file_reads, args.samples // 3, args.reps)
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as fh:
            fh.write(text + '\n')


if __name__ == '__main__':
    main()
