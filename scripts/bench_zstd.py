"""zstd frames decoded on the device: kernel rate against libzstd on every host core, the end-to-end call from
frames against the same reads from post-zstd bodies, and fast5 files to overview.csv with zstd on the device
against zstd on the host.

    python scripts/bench_zstd.py --out profiles/r05_zstd.json

(a) wstr_zstd_decode_batch alone: --frames level-1 frames of --chunk-sample chunks of synthetic HD reads
    (synth.to_raw_int16, VBZ v0 bodies), --pool distinct ones repeated at distinct addresses (input and output
    far above the 126 MB L2), CUDA events over --passes launches after a warm-up.  libzstd (ctypes, GIL
    released) decodes the same frames on a thread per host core in the same run.
(b) CallerEngine.call_arrays_vbz on the same reads (HD locus) packed from frames and from post-zstd bodies,
    alternated: reads/s and bytes across PCIe.
(c) main_wrapper on multi-read fast5 files (tests/_h5write.py), zstd on the device (fast5.stored_chunks)
    against zstd on the host (fast5.raw_chunks), wall clock; host parse time of each workload reported apart.
"""
import argparse
import ctypes
import json
import os
import shutil
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
sys.path.insert(0, os.path.join(ROOT, 'scripts'))

from bench_vbz import card, events_ms  # noqa: E402


def _frames_of(comp):
    """CompressedReads of bodies -> the same reads with every VBZ body as a level-1 zstd frame."""
    import _zstd as Z
    from warpstr_b200 import fast5
    out = []
    for r in comp:
        ch = [c._replace(kind=c.kind + fast5.KIND_VBZ0_ZSTD, payload=Z.compress(c.payload, 1), body_size=len(c.payload))
              if c.kind != fast5.KIND_RAW else c for c in r.chunks]
        out.append(fast5.CompressedRead(r.path, r.read_name, r.n_samples, ch))
    return out


def bench_kernel(args):
    import _h5write as hw
    import _zstd as Z
    import torch
    from warpstr_b200 import _lib
    x = Z.synthetic_raw(args.pool * args.chunk_samples, seed=11)
    bodies = [hw.svb_body(x[i * args.chunk_samples:(i + 1) * args.chunk_samples], 0) for i in range(args.pool)]
    frames = [Z.compress(b, 1) for b in bodies]
    reps = (args.frames + args.pool - 1) // args.pool
    n = args.pool * reps
    fb = np.array([len(f) for f in frames] * reps, dtype=np.int64)
    ob = np.array([len(b) for b in bodies] * reps, dtype=np.int64)
    in_off = np.zeros(n, dtype=np.int64)
    in_off[1:] = np.cumsum((fb[:-1] + 15) & ~15)
    out_off = np.zeros(n, dtype=np.int64)
    out_off[1:] = np.cumsum((ob[:-1] + 15) & ~15)
    pool_pay = np.zeros(int(((fb[:args.pool] + 15) & ~15).sum()), dtype=np.uint8)
    for f, o in zip(frames, in_off[:args.pool]):
        pool_pay[o:o + len(f)] = np.frombuffer(f, dtype=np.uint8)
    d_in = torch.from_numpy(pool_pay).cuda().repeat(reps)
    d_out = torch.empty(int(out_off[-1] + ob[-1]), dtype=torch.uint8, device='cuda')
    d_st = torch.empty(n, dtype=torch.int32, device='cuda')
    ws = torch.empty(_lib.zstd_workspace_bytes(n), dtype=torch.uint8, device='cuda')

    def run():
        _lib.zstd_decode_batch(d_in, in_off, fb, out_off, ob, d_out, d_st, ws)
    ms = events_ms(run, args.passes)
    assert not d_st.any().item()
    for k in (0, n - 1):
        got = d_out[int(out_off[k]):int(out_off[k] + ob[k])].cpu().numpy().tobytes()
        assert got == bodies[k % args.pool]
    out_bytes, in_bytes = int(ob.sum()), int(fb.sum())
    # libzstd on every host core, the same frames
    z = Z.lib()
    cap = int(ob.max())

    def host_part(ks):
        buf = ctypes.create_string_buffer(cap)
        for k in ks:
            f = frames[k % args.pool]
            assert z.ZSTD_decompress(buf, cap, f, len(f)) == len(bodies[k % args.pool])
    cores = os.cpu_count()
    parts = np.array_split(np.arange(n), cores)
    with ThreadPoolExecutor(cores) as ex:
        list(ex.map(host_part, [p[:8] for p in parts]))                  # warm-up
        t0 = time.perf_counter()
        list(ex.map(host_part, parts))
        host_s = time.perf_counter() - t0
    return dict(frames=n, distinct=args.pool, chunk_samples=args.chunk_samples, level=1, input_bytes=in_bytes,
                output_bytes=out_bytes, ms=ms, frames_per_s=n / ms * 1e3, output_gbs=out_bytes / ms / 1e6,
                input_gbs=in_bytes / ms / 1e6, host_cores=cores, libzstd_all_cores_s=host_s,
                libzstd_output_gbs=out_bytes / host_s / 1e9, libzstd_frames_per_s=n / host_s,
                includes='frame-table staging in every launch; libzstd decodes --pool distinct frames (cache-warm)')


def bench_e2e(args):
    import torch
    from bench_vbz import compress
    from warpstr_b200 import synth
    from warpstr_b200.automata import StateAutomata
    from warpstr_b200.caller import CallerEngine, pack_vbz
    locus = synth.make_locus('HD', seed=1)
    stas = [StateAutomata(locus.template_regex), StateAutomata(locus.reverse_regex)]
    reads = synth.make_reads(locus, args.e2e_pool, seed=2)
    rng = np.random.default_rng(3)
    raws, wins = [], []
    for r in reads:
        pad = max(args.samples - len(r.signal), 2000) // 2
        raw, lo, hi = synth.to_raw_int16(rng, r.signal, pad=pad, spike_rate=1e-4)
        raws.append(raw)
        wins.append((lo, hi))
    reps = (args.e2e_reads + args.e2e_pool - 1) // args.e2e_pool
    raws, wins = raws * reps, wins * reps
    rev = np.array([r.reverse for r in reads] * reps, dtype=np.uint8)
    eng = CallerEngine()
    ids = [eng.add_automaton(s, locus.flank_length) for s in stas]
    aut = np.array([ids[int(x)] for x in rev], dtype=np.int32)
    bodies = compress(raws[:args.e2e_pool], args.chunk_samples)
    packs = {'bodies': pack_vbz(bodies * reps), 'frames': pack_vbz(_frames_of(bodies) * reps)}
    lo, hi = [w[0] for w in wins], [w[1] for w in wins]
    runs = {k: (lambda p=p: eng.call_arrays_vbz(p[0], p[1], p[2], p[3], lo, hi, aut, rev, 'Brute'))
            for k, p in packs.items()}
    first = {k: {kk: (v.copy() if isinstance(v, np.ndarray) else v) for kk, v in f().items()} for k, f in runs.items()}
    assert not first['frames']['zstd_status'].any()
    for k in ('len1', 'len2', 'cost1', 'cost2', 'status', 'shift_scale'):
        assert np.array_equal(first['bodies'][k], first['frames'][k], equal_nan=True), k
    times = {k: [] for k in runs}
    for _ in range(args.e2e_rounds):
        for k, f in runs.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            f()
            torch.cuda.synchronize()
            times[k].append(time.perf_counter() - t0)
    n = len(raws)
    return dict(reads=n, samples=int(sum(len(x) for x in raws)), locus='HD',
                **{k: dict(s=times[k], reads_per_s=n / float(np.median(times[k])), h2d_bytes=int(packs[k][0].numel()))
                   for k in runs})


def bench_files(args):
    import _h5write as hw
    import torch
    from warpstr_b200 import caller_only, fast5, synth
    from warpstr_b200.overview import load_overview
    from warpstr_b200.wrapper import CallerWrapper, Locus, flanks_from_template, get_compressed_workload, main_wrapper
    tmp = tempfile.mkdtemp(prefix='bench_zstd_')
    stored = fast5.stored_chunks
    try:
        locus = synth.make_locus('HD', seed=5)
        reads = synth.make_reads(locus, args.file_reads, seed=6)
        rng = np.random.default_rng(7)
        rows, files, batch = [], [], {}
        for i, r in enumerate(reads):
            pad = max(args.samples - len(r.signal), 2000) // 2
            raw, lo, hi = synth.to_raw_int16(rng, r.signal, pad=pad, spike_rate=1e-4)
            rid = f'{i:06d}-bench'
            batch[rid] = raw
            rows.append((len(files), rid, r.reverse, lo, hi))
            if len(batch) == args.reads_per_file or i == len(reads) - 1:
                p = os.path.join(tmp, f'batch{len(files)}.fast5')
                hw.write_multi(p, batch, 'vbz0', chunk=args.chunk_samples)
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
        def host_zstd(path, read_name=None, h5=None):
            r = stored(path, read_name, h5)
            r.chunks = [c.unzstd() for c in r.chunks]
            return r
        routes = {'host_zstd': host_zstd, 'device_zstd': stored}
        t = {f'{k}_{w}': [] for k in routes for w in ('main_wrapper_s', 'parse_s')}
        outs = {}
        for rnd in range(args.file_rounds + 1):                              # round 0 warms up
            for k, fn in routes.items():
                fast5.stored_chunks = fn
                open(os.path.join(d, 'overview.csv'), 'wb').write(pristine)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                main_wrapper(loc, flanks=flanks, engine=cw.engine)
                t1 = time.perf_counter()
                get_compressed_workload(df, d)
                t2 = time.perf_counter()
                outs[k] = open(os.path.join(d, 'overview.csv'), 'rb').read()
                if rnd:
                    t[f'{k}_main_wrapper_s'].append(t1 - t0)
                    t[f'{k}_parse_s'].append(t2 - t1)
        assert outs['host_zstd'] == outs['device_zstd']
        med = {k: float(np.median(v)) for k, v in t.items()}
        return dict(reads=len(reads), files=len(files), chunk_samples=args.chunk_samples, seconds=t, median=med,
                    speedup=med['host_zstd_main_wrapper_s'] / med['device_zstd_main_wrapper_s'],
                    host_cpus=os.cpu_count())
    finally:
        fast5.stored_chunks = stored
        shutil.rmtree(tmp, ignore_errors=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--frames', type=int, default=40000)
    ap.add_argument('--pool', type=int, default=64, help='distinct frames, repeated to --frames')
    ap.add_argument('--chunk-samples', type=int, default=102400)
    ap.add_argument('--passes', type=int, default=5)
    ap.add_argument('--samples', type=int, default=150000)
    ap.add_argument('--e2e-pool', type=int, default=200)
    ap.add_argument('--e2e-reads', type=int, default=10000)
    ap.add_argument('--e2e-rounds', type=int, default=5)
    ap.add_argument('--file-reads', type=int, default=2000)
    ap.add_argument('--reads-per-file', type=int, default=500)
    ap.add_argument('--file-rounds', type=int, default=3)
    ap.add_argument('--skip', default='', help='comma list of kernel,e2e,files')
    ap.add_argument('--out', default='')
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('bench_zstd.py needs a CUDA device')
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
