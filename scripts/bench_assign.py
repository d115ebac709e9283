"""Measure the flank assignment (DESIGN.md section 4.6) on one GPU: writes <out>/r07_assign.{json,md}.

* Panels of 1, 10 and 50 synthetic loci (four 105-state flank chains each) against whole reads of ~150 000
  normalised samples of random sequence (a read's cost does not depend on what it carries): reads/s, cells/s
  (cells = samples x chain states) and their ratio to the same run's wstr_measure_fp64_add_rate.
* The gain from grouping: wstr_assign_batch (locate_group_kernel, all chains of a read in few CTAs) against
  wstr_locate_batch (locate_kernel, one CTA per (read, chain)) on the same entries.
* Files to overviews: assign.assign_files on a POD5 file of whole reads (host read, upload, zstd / VBZ decode,
  normalisation, search, overview CSV).

    python scripts/bench_assign.py [--reads 10000,2000,400] [--file-reads 500] [--out profiles]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else 'unknown'


def make_reads(torch, n, length, seed, device):
    """n reads of length - U{0..1999} samples: pore levels of random 6-mers, dwell U{5..13}, noise 0.15."""
    from warpstr_b200 import synth
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    lengths = (length - torch.randint(0, 2000, (n,), generator=g, device=device)).cpu().numpy().astype(np.int32)
    padded = (lengths.astype(np.int64) + 1) & ~1
    off = np.zeros(n, dtype=np.int64)
    off[1:] = np.cumsum(padded[:-1])
    total = int(padded.sum())
    table = torch.from_numpy(synth.get_pore_model().table).to(device)
    k = total // 9 + 16
    lev = table[torch.randint(0, len(table), (k,), generator=g, device=device)]
    dw = torch.randint(5, 14, (k,), generator=g, device=device)
    sig = torch.repeat_interleave(lev, dw)[:total]
    sig = sig + 0.15 * torch.randn(total, generator=g, device=device, dtype=torch.float64)
    return sig.contiguous(), off, lengths


def panel(n_loci, seed=7):
    from warpstr_b200 import synth
    from warpstr_b200.assign import Panel
    from warpstr_b200.wrapper import flanks_from_template
    loci = synth.make_panel(n_loci, seed=seed)
    return loci, Panel([(L.name, flanks_from_template(L.left, L.right)) for L in loci])


def timed(torch, fn, reps=1):
    fn()                                             # warm-up: module load, buffers
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / 1e3 / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reads', default='10000,2000,400', help='reads for the 1-, 10- and 50-locus panels')
    ap.add_argument('--length', type=int, default=150_000)
    ap.add_argument('--pair-reads', type=int, default=200, help='reads of the grouped / per-entry comparison')
    ap.add_argument('--file-reads', type=int, default=500)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles'))
    args = ap.parse_args()
    import torch
    from warpstr_b200 import _lib
    from warpstr_b200.caller import CallerEngine
    assert torch.cuda.is_available(), 'bench_assign needs a GPU'
    dev = torch.device('cuda')
    # wstr_measure_fp64_add_rate gives 10^12 FP64 adds per second
    res = dict(gpu=gpu_info(), length=args.length, fp64_adds_per_s=_lib.measure_fp64_add_rate() * 1e12, panels=[])
    print(res['gpu'], f"fp64 adds {res['fp64_adds_per_s']:.3e}/s")
    for n_loci, n in zip((1, 10, 50), (int(x) for x in args.reads.split(','))):
        eng = CallerEngine()
        _, pan = panel(n_loci)
        d_sig, off, lengths = make_reads(torch, n, args.length, 11 + n_loci, dev)
        states = sum(c.n_states for c in pan.chains)
        t = timed(torch, lambda: eng.assign_packed(d_sig, off, lengths, pan))
        cells = float(lengths.astype(np.int64).sum()) * states
        row = dict(loci=n_loci, reads=n, chain_states=states, seconds=t, reads_per_s=n / t, cells_per_s=cells / t,
                   cells_per_fp64_add=cells / t / res['fp64_adds_per_s'])
        # grouped against per-entry on the same (read, chain) entries
        m = min(args.pair_reads, n)
        ids = pan.register(eng)
        auts = [eng.automata[i] for i in ids]
        A = len(auts)
        sub_off, sub_len = off[:m], lengths[:m]
        tg = timed(torch, lambda: eng.assign_packed(d_sig, sub_off, sub_len, pan))
        ra = np.tile(np.arange(A, dtype=np.int32), m)
        rd = np.repeat(np.arange(m), A)
        d_i = torch.empty((3, m * A), dtype=torch.int32, device=dev)
        d_sc = torch.empty(m * A, dtype=torch.float64, device=dev)
        lws = torch.empty(_lib.locate_workspace_bytes(auts, m * A), dtype=torch.uint8, device=dev)
        tl = timed(torch, lambda: _lib.locate_batch(auts, ra, d_sig, sub_off[rd], sub_len[rd], 0.35, d_i[0], d_i[1],
                                                    d_sc, d_i[2], lws))
        row.update(pair_reads=m, grouped_s=tg, per_entry_s=tl, grouping_gain=tl / tg)
        print(json.dumps(row))
        res['panels'].append(row)
        del d_sig, eng
        torch.cuda.empty_cache()
    # files -> overviews from POD5
    import _pod5write as pw
    import uuid
    from warpstr_b200 import synth
    from warpstr_b200.assign import assign_files
    from warpstr_b200.config import Config, LocusConfig
    from warpstr_b200.wrapper import flanks_from_template
    loci, _ = panel(10)
    rng = np.random.default_rng(5)
    d_sig, off, lengths = make_reads(torch, args.file_reads, args.length, 99, dev)
    host = d_sig.cpu().numpy()
    reads = {str(uuid.UUID(bytes=rng.bytes(16), version=4)):
             np.rint((90.8717 + 9.8354 * host[o:o + L]) * 5.85).astype(np.int16) for o, L in zip(off, lengths)}
    del d_sig
    with tempfile.TemporaryDirectory() as tmp:
        p5 = os.path.join(tmp, 'run.pod5')
        pw.write(p5, reads, rows=1)
        cfg = Config(output=os.path.join(tmp, 'out'), loci=[LocusConfig(name=L.name, sequence=L.sequence) for L in loci])
        flanks = {L.name: flanks_from_template(L.left, L.right) for L in loci}
        eng = CallerEngine()
        assign_files(cfg, [p5], engine=eng, flanks=flanks, verbose=False)        # warm-up
        t0 = time.perf_counter()
        assign_files(cfg, [p5], engine=eng, flanks=flanks, verbose=False)
        torch.cuda.synchronize()
        tf = time.perf_counter() - t0
    res['files'] = dict(loci=10, reads=args.file_reads, seconds=tf, reads_per_s=args.file_reads / tf)
    print(json.dumps(res['files']))
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, 'r07_assign.json'), 'w') as fh:
        json.dump(res, fh, indent=1)
    lines = [f"# Flank assignment (scripts/bench_assign.py)", '', f"GPU: {res['gpu']} (name, power limit, max SM clock, "
             f"read in the same run).  wstr_measure_fp64_add_rate: {res['fp64_adds_per_s']:.3e} adds/s.", '',
             '| loci | chain states | reads | s | reads/s | cells/s | cells / fp64 add | grouped vs per-entry '
             '(reads) |', '|---|---|---|---|---|---|---|---|']
    for r in res['panels']:
        lines.append(f"| {r['loci']} | {r['chain_states']} | {r['reads']} | {r['seconds']:.2f} | {r['reads_per_s']:.0f} "
                     f"| {r['cells_per_s']:.3e} | {r['cells_per_fp64_add']:.4f} | {r['grouping_gain']:.2f}x "
                     f"({r['pair_reads']}) |")
    f = res['files']
    lines += ['', f"Files to overviews (assign_files, 10-locus panel, one POD5 file of {f['reads']} reads of "
              f"~{args.length} samples): {f['seconds']:.2f} s, {f['reads_per_s']:.0f} reads/s."]
    with open(os.path.join(args.out, 'r07_assign.md'), 'w') as fh:
        fh.write('\n'.join(lines) + '\n')


if __name__ == '__main__':
    main()
