"""The same reads from POD5 files and from fast5 files: host parse time per read of each container, and
main_wrapper from files to overview.csv on the GPU for each.

    python scripts/bench_pod5.py --out profiles/r06_pod5.json            # on a GPU machine
    python scripts/bench_pod5.py --parse-only --out /tmp/parse.json      # host parse only, no GPU needed

--reads synthetic HD reads (synth.to_raw_int16, --samples samples each) go into files of --reads-per-file reads,
written twice with the test writers: POD5 (tests/_pod5write.py: one level-1 zstd frame of VBZ v1 per signal row,
rows of at most --row-samples samples, as MinKNOW cuts them, scattered over the signal table) and multi-read fast5
(tests/_h5write.py: VBZ v1 with zstd level 1 in chunks of --row-samples).  Both code the same StreamVByte bodies,
so the device chain after the parse is the same work.

(a) parse: ``wrapper.get_compressed_workload`` on each container's overview (every file opened and indexed once,
    every read's chunks as stored), wall clock, --rounds rounds after a warm-up, medians; reported per read.
(b) main_wrapper, files to overview.csv, the two containers alternated, --rounds rounds after a warm-up, medians;
    the overviews must agree but for the source column's paths.  The card's name and power limit are read in the
    same run.
"""
import argparse
import json
import os
import shutil
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
sys.path.insert(0, os.path.join(ROOT, 'scripts'))


def write_files(args, tmp):
    """-> (locus, overview dirs {container: dir}, bytes on disk {container: n})."""
    import uuid
    import _h5write as hw
    import _pod5write as pw
    from warpstr_b200 import caller_only, synth
    locus = synth.make_locus('HD', seed=5)
    rng = np.random.default_rng(7)
    rows, dirs, size = [], {}, {'pod5': 0, 'fast5': 0}
    n_files = (args.reads + args.reads_per_file - 1) // args.reads_per_file
    for f in range(n_files):
        n = min(args.reads_per_file, args.reads - f * args.reads_per_file)
        reads = synth.make_reads(locus, n, seed=100 + f)
        batch = {}
        for r in reads:
            pad = max(args.samples - len(r.signal), 2000) // 2
            raw, lo, hi = synth.to_raw_int16(rng, r.signal, pad=pad, spike_rate=1e-4)
            rid = str(uuid.UUID(bytes=rng.bytes(16)))
            batch[rid] = raw
            rows.append((f, rid, r.reverse, lo, hi))
        p = os.path.join(tmp, f'batch{f}')
        pw.write(p + '.pod5', batch, rows=lambda k, m: -(-m // args.row_samples), seed=f, shuffle=True)
        hw.write_multi(p + '.fast5', batch, 'vbz1', chunk=args.row_samples)
        for c in size:
            size[c] += os.path.getsize(f'{p}.{c}')
    for c in ('pod5', 'fast5'):
        csv_path = os.path.join(tmp, f'reads_{c}.csv')
        with open(csv_path, 'w') as fh:
            fh.write('fast5_path,locus,read_name,reverse,l_start_raw,r_end_raw\n')
            for f, rid, rv, lo, hi in rows:
                fh.write(f'{os.path.join(tmp, f"batch{f}.{c}")},LOC,{rid},{rv},{lo},{hi}\n')
        caller_only.prepare(os.path.join(tmp, f'out_{c}'), csv_path)
        dirs[c] = os.path.join(tmp, f'out_{c}', 'LOC')
    return locus, dirs, size


def bench_parse(args, dirs):
    from warpstr_b200.overview import load_overview
    from warpstr_b200.wrapper import get_compressed_workload
    t = {c: [] for c in dirs}
    for rnd in range(args.rounds + 1):                                   # round 0 warms the page cache
        for c, d in dirs.items():
            _, df = load_overview(d)
            t0 = time.perf_counter()
            reads = get_compressed_workload(df, d)[2]
            t1 = time.perf_counter()
            if rnd:
                t[c].append(t1 - t0)
    n = len(reads)
    med = {c: float(np.median(v)) for c, v in t.items()}
    return dict(reads=n, seconds=t, median_s=med, us_per_read={c: 1e6 * v / n for c, v in med.items()},
                pod5_over_fast5=med['pod5'] / med['fast5'])


def bench_main_wrapper(args, locus, dirs):
    import torch
    from warpstr_b200.wrapper import CallerWrapper, Locus, flanks_from_template, main_wrapper
    flanks = flanks_from_template(locus.left, locus.right)
    locs = {c: Locus(name='LOC', sequence=locus.sequence, flank_length=locus.flank_length, path=d)
            for c, d in dirs.items()}
    engine = CallerWrapper(locs['pod5'], flanks=flanks).engine
    pristine = {c: open(os.path.join(d, 'overview.csv'), 'rb').read() for c, d in dirs.items()}
    t = {c: [] for c in dirs}
    outs = {}
    for rnd in range(args.rounds + 1):                                   # round 0 warms up
        for c, d in dirs.items():
            open(os.path.join(d, 'overview.csv'), 'wb').write(pristine[c])
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            main_wrapper(locs[c], flanks=flanks, engine=engine)
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            outs[c] = open(os.path.join(d, 'overview.csv'), 'rb').read()
            if rnd:
                t[c].append(t1 - t0)
    same = outs['pod5'].replace(b'.pod5', b'.fast5') == outs['fast5']
    assert same, 'the two containers gave different overviews'
    med = {c: float(np.median(v)) for c, v in t.items()}
    return dict(seconds=t, median_s=med, reads_per_s={c: args.reads / v for c, v in med.items()},
                pod5_over_fast5=med['pod5'] / med['fast5'], overviews_agree=same)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reads', type=int, default=10000)
    ap.add_argument('--samples', type=int, default=150000)
    ap.add_argument('--reads-per-file', type=int, default=2500)
    ap.add_argument('--row-samples', type=int, default=102400)
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--parse-only', action='store_true', help='host parse only (no GPU needed)')
    ap.add_argument('--out', default='')
    args = ap.parse_args()
    res = {'args': {k: v for k, v in vars(args).items() if k != 'out'}, 'host_cpus': os.cpu_count()}
    if not args.parse_only:
        import torch
        if not torch.cuda.is_available():
            raise SystemExit('bench_pod5.py needs a CUDA device (or --parse-only)')
        import __graft_entry__ as ge
        if not os.path.exists(ge.LIB):
            raise SystemExit('build first: python -c "import __graft_entry__ as g; g.build()"')
        from bench_vbz import card
        res['card'] = card()
    tmp = tempfile.mkdtemp(prefix='bench_pod5_')
    try:
        t0 = time.perf_counter()
        locus, dirs, size = write_files(args, tmp)
        res['files'] = dict(bytes=size, write_s=time.perf_counter() - t0)
        print(json.dumps({'files': res['files']}), flush=True)
        res['parse'] = bench_parse(args, dirs)
        print(json.dumps({'parse': res['parse']}), flush=True)
        if not args.parse_only:
            res['main_wrapper'] = bench_main_wrapper(args, locus, dirs)
            print(json.dumps({'main_wrapper': res['main_wrapper']}), flush=True)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as fh:
            json.dump(res, fh, indent=1)


if __name__ == '__main__':
    main()
