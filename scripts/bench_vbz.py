"""VBZ decoding on the device: kernel rate, the end-to-end call from pinned host memory against the int16
route, and fast5 files to overview.csv against the host-decode route.

    python scripts/bench_vbz.py --out profiles/r03_vbz.json

1. wstr_vbz_decode_batch alone, CUDA events over --passes launches after a warm-up, on --reads reads of
   --samples samples in chunks of --chunk (payload + int16 output far above the 126 MB L2).  Bytes counted:
   payload read + int16 written.  Share of HBM against the measured 6.55 TB/s DESIGN §4.2 uses for the
   normalisation kernel, and against a device-to-device copy timed in the same run.
2. CallerEngine.call_arrays_vbz against call_arrays_raw on the same reads (HD locus, whole reads of
   ~--samples samples), alternated, from pinned host memory: reads/s and bytes across PCIe.
3. main_wrapper on --file-reads reads in multi-read fast5 files (tests/_h5write.py) against the previous
   route (get_raw_workload + CallerWrapper.run_raw), wall clock; host seconds per read of parsing + zstd.
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

HBM_MEASURED_GBS = 6550.0     # DESIGN §4.2's denominator (measured HBM peak of the B200)


def card():
    import torch
    out = {'name': torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        out['nvidia_smi'] = q[0] if q else ''
    except (OSError, subprocess.SubprocessError) as exc:
        out['nvidia_smi'] = f'unavailable: {exc}'
    return out


def pool_reads(n_pool, samples, seed):
    """Nanopore-like int16 reads: a random walk around a level, some spikes."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n_pool):
        n = int(rng.integers(int(samples * 0.9), int(samples * 1.1)))
        x = 480 + np.cumsum(rng.normal(0, 6, size=n)) * 0.1 + rng.normal(0, 12, size=n)
        out.append(np.clip(x, -32768, 32767).astype(np.int16))
    return out


def compress(reads, chunk, version=0):
    import _h5write as hw
    from warpstr_b200 import fast5
    comp = []
    for i, x in enumerate(reads):
        chunks = [fast5.RawChunk(s, len(x[s:s + chunk]), version, hw.svb_body(x[s:s + chunk], version, True), True,
                                 len(x[s:s + chunk])) for s in range(0, len(x), chunk)]
        comp.append(fast5.CompressedRead('bench', str(i), len(x), chunks))
    return comp


def events_ms(fn, passes, warmup=3):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(passes):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / passes


def bench_kernel(args):
    import torch
    from warpstr_b200 import _lib
    from warpstr_b200.caller import pack_vbz
    pool = pool_reads(args.pool, args.samples, 1)
    host, table, read_chunk, raw_off = pack_vbz(compress(pool, args.chunk))
    reps = (args.reads + args.pool - 1) // args.pool
    pool_bytes, pool_samples, m = host.numel(), int(raw_off[-1]), len(table['in_off'])
    d_payload = host.cuda().repeat(reps)                        # distinct copies: nothing is served from L2
    t = {k: np.concatenate([v + (pool_bytes * r if k == 'in_off' else pool_samples * r if k == 'out_off' else 0)
                            for r in range(reps)]) for k, v in table.items()}
    n_chunks = len(t['in_off'])
    d_raw = torch.empty(pool_samples * reps + 8, dtype=torch.int16, device='cuda')
    d_status = torch.empty(n_chunks, dtype=torch.int32, device='cuda')
    ws = torch.empty(_lib.vbz_workspace_bytes(n_chunks), dtype=torch.uint8, device='cuda')

    def run():
        _lib.vbz_decode_batch(d_payload, t['in_off'], t['in_bytes'], t['n_samples'], t['n_out'], t['kind'],
                              t['zigzag'], t['out_off'], d_raw, d_status, ws)
    ms = events_ms(run, args.passes)
    assert not d_status.any().item()
    # spot check against the host decoder
    got = d_raw[int(raw_off[3]):int(raw_off[4])].cpu().numpy()
    assert np.array_equal(got, pool[3])
    samples = pool_samples * reps
    moved = int(t['in_bytes'].sum()) + 2 * samples
    src = torch.empty(moved // 2, dtype=torch.uint8, device='cuda')
    dst = torch.empty_like(src)
    copy_ms = events_ms(lambda: dst.copy_(src), args.passes)
    copy_gbs = 2 * src.numel() / copy_ms / 1e6
    gbs = moved / ms / 1e6
    return dict(reads=args.pool * reps, samples=samples, chunks=n_chunks, chunk_samples=args.chunk,
                payload_bytes_per_sample=int(t['in_bytes'].sum()) / samples, ms=ms, samples_per_s=samples / ms * 1e3,
                gbs=gbs, hbm_fraction_measured_peak=gbs / HBM_MEASURED_GBS, d2d_copy_gbs=copy_gbs,
                fraction_of_d2d_copy=gbs / copy_gbs, includes='chunk-table staging (upload_kernel) in every launch')


def bench_e2e(args):
    import torch
    from warpstr_b200 import synth
    from warpstr_b200.automata import StateAutomata
    from warpstr_b200.caller import CallerEngine, pack_vbz
    locus = synth.make_locus('HD', seed=1)
    stas = [StateAutomata(locus.template_regex), StateAutomata(locus.reverse_regex)]
    reads = synth.make_reads(locus, args.pool, seed=2)
    rng = np.random.default_rng(3)
    raws, wins = [], []
    for r in reads:
        pad = max(args.samples - len(r.signal), 2000) // 2
        raw, lo, hi = synth.to_raw_int16(rng, r.signal, pad=pad, spike_rate=1e-4)
        raws.append(raw)
        wins.append((lo, hi))
    reps = (args.e2e_reads + args.pool - 1) // args.pool
    raws, wins = raws * reps, wins * reps
    rev = np.array([r.reverse for r in reads] * reps, dtype=np.uint8)
    eng = CallerEngine()
    ids = [eng.add_automaton(s, locus.flank_length) for s in stas]
    aut = np.array([ids[int(x)] for x in rev], dtype=np.int32)
    roff = np.zeros(len(raws) + 1, dtype=np.int64)
    roff[1:] = np.cumsum([len(x) for x in raws])
    hraw = torch.from_numpy(np.concatenate(raws)).pin_memory()
    host, table, read_chunk, raw_off = pack_vbz(compress(raws[:args.pool], args.chunk) * reps)
    assert np.array_equal(raw_off, roff)
    lo, hi = [w[0] for w in wins], [w[1] for w in wins]
    runs = {'raw': lambda: eng.call_arrays_raw(hraw, roff, lo, hi, aut, rev, 'Brute'),
            'vbz': lambda: eng.call_arrays_vbz(host, table, read_chunk, raw_off, lo, hi, aut, rev, 'Brute')}
    first = {k: {kk: (v.copy() if isinstance(v, np.ndarray) else v) for kk, v in f().items()} for k, f in runs.items()}
    for k in ('len1', 'len2', 'cost1', 'cost2', 'status', 'shift_scale'):
        assert np.array_equal(first['raw'][k], first['vbz'][k], equal_nan=True), k
    times = {k: [] for k in runs}
    for _ in range(args.e2e_rounds):
        for k, f in runs.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            f()
            torch.cuda.synchronize()
            times[k].append(time.perf_counter() - t0)
    n = len(raws)
    return dict(reads=n, samples=int(roff[-1]), locus='HD',
                raw=dict(s=times['raw'], reads_per_s=n / float(np.median(times['raw'])), h2d_bytes=int(roff[-1]) * 2),
                vbz=dict(s=times['vbz'], reads_per_s=n / float(np.median(times['vbz'])),
                         h2d_bytes=int(host.numel())))


def bench_files(args):
    import _h5write as hw
    import torch
    from warpstr_b200 import caller_only, synth
    from warpstr_b200.overview import load_overview
    from warpstr_b200.wrapper import (CallerWrapper, Locus, flanks_from_template, get_compressed_workload,
                                      get_raw_workload, main_wrapper)
    tmp = tempfile.mkdtemp(prefix='bench_vbz_')
    try:
        locus = synth.make_locus('HD', seed=5)
        reads = synth.make_reads(locus, args.file_reads, seed=6)
        rng = np.random.default_rng(7)
        per_file = args.reads_per_file
        rows, files = [], []
        batch = {}
        for i, r in enumerate(reads):
            pad = max(args.samples - len(r.signal), 2000) // 2
            raw, lo, hi = synth.to_raw_int16(rng, r.signal, pad=pad, spike_rate=1e-4)
            rid = f'{i:06d}-bench'
            batch[rid] = raw
            rows.append((len(files), rid, r.reverse, lo, hi))
            if len(batch) == per_file or i == len(reads) - 1:
                p = os.path.join(tmp, f'batch{len(files)}.fast5')
                hw.write_multi(p, batch, 'vbz0', chunk=args.file_chunk)
                files.append(p)
                batch = {}
        csv_path = os.path.join(tmp, 'reads.csv')
        with open(csv_path, 'w') as fh:
            fh.write('fast5_path,locus,read_name,reverse,l_start_raw,r_end_raw\n')
            for k, rid, rv, lo, hi in rows:
                fh.write(f'{files[k]},LOC,{rid},{rv},{lo},{hi}\n')
        caller_only.prepare(os.path.join(tmp, 'out'), csv_path)
        d = os.path.join(tmp, 'out', 'LOC')
        loc = Locus(name='LOC', sequence=locus.sequence, flank_length=locus.flank_length, path=d)
        flanks = flanks_from_template(locus.left, locus.right)
        cw = CallerWrapper(loc, flanks=flanks)
        pristine = open(os.path.join(d, 'overview.csv'), 'rb').read()
        _, df = load_overview(d)
        main_wrapper(loc, flanks=flanks, engine=cw.engine)                    # warm-up
        t = {'previous': [], 'main_wrapper': [], 'parse_zstd': []}
        for _ in range(args.file_rounds):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            names, revs, raws, wins = get_raw_workload(df, d)
            res_prev = cw.run_raw(raws, wins, revs)
            t['previous'].append(time.perf_counter() - t0)
            open(os.path.join(d, 'overview.csv'), 'wb').write(pristine)
            t0 = time.perf_counter()
            main_wrapper(loc, flanks=flanks, engine=cw.engine)
            t['main_wrapper'].append(time.perf_counter() - t0)
            t0 = time.perf_counter()
            get_compressed_workload(df, d)
            t['parse_zstd'].append(time.perf_counter() - t0)
        names, revs, comp, wins = get_compressed_workload(df, d)
        assert res_prev == cw.run_compressed(comp, wins, revs)
        n = len(reads)
        med = {k: float(np.median(v)) for k, v in t.items()}
        return dict(reads=n, files=len(files), samples=int(sum(len(x) for x in raws)), chunk_samples=args.file_chunk,
                    seconds=t, previous_s=med['previous'], main_wrapper_s=med['main_wrapper'],
                    speedup=med['previous'] / med['main_wrapper'], host_parse_zstd_s_per_read=med['parse_zstd'] / n,
                    host_cpus=os.cpu_count())
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reads', type=int, default=20000)
    ap.add_argument('--samples', type=int, default=150000)
    ap.add_argument('--chunk', type=int, default=102400, help='samples per HDF5 chunk')
    ap.add_argument('--pool', type=int, default=200, help='distinct reads, repeated to the batch size')
    ap.add_argument('--passes', type=int, default=20)
    ap.add_argument('--e2e-reads', type=int, default=10000)
    ap.add_argument('--e2e-rounds', type=int, default=5)
    ap.add_argument('--file-reads', type=int, default=2000)
    ap.add_argument('--reads-per-file', type=int, default=500)
    ap.add_argument('--file-chunk', type=int, default=102400)
    ap.add_argument('--file-rounds', type=int, default=3)
    ap.add_argument('--skip', default='', help='comma list of kernel,e2e,files')
    ap.add_argument('--out', default='')
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('bench_vbz.py needs a CUDA device')
    import __graft_entry__ as ge
    if not os.path.exists(ge.LIB):
        raise SystemExit('build first: python -c "import __graft_entry__ as g; g.build()"')
    res = {'card': card(), 'args': {k: v for k, v in vars(args).items() if k != 'out'}}
    skip = set(args.skip.split(','))
    for name, fn in (('kernel', bench_kernel), ('e2e', bench_e2e), ('files', bench_files)):
        if name not in skip:
            res[name] = fn(args)
            print(json.dumps({name: res[name]}), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as fh:
            json.dump(res, fh, indent=1)


if __name__ == '__main__':
    main()
