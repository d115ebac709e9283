#!/usr/bin/env python
"""Benchmark of the WarpSTR caller hot path on B200.

  python bench.py --gpus N --steps K --warmup W            (N>1: launched under torchrun)
  python bench.py --impl reference --gpus N --steps K --warmup W
  python bench.py ... --dump-outputs DIR                   (also writes the results of the last timed step, see
                                                           dump_outputs: the inputs depend on the arguments only)

Workload (BASELINE.json configs[1], SURVEY.md section 8d C2): a synthetic batch of HD-locus reads
`(AGC)AACAGCCGCCAC(CGC)`, AGC~U{30..45}, CGC~U{7..12}, 50 % reverse strand, dwell U{5..13},
noise N(0, 0.15), float64, ~3.3 k samples per read, 100 000 reads per GPU (weak scaling: every
rank gets its own 100 000 reads and its own seed; the per-read results are gathered every step).

One step = the whole per-read call (two DP passes + everything between them) over the batch.
  value        reads/s with the batch resident in HBM (wstr_call_batch on device buffers)
  e2e          reads/s from pinned host memory to host result arrays, every step: the batch as int16 window
               samples + {shift, scale} per read (CallerEngine.call_arrays_quantized); e2e_float64 is the same
               call on float64 windows (the reference's ReadSignal.signal), e2e_raw whole raw reads in
               (normalised on the device)
  roofline     the DP fill+traceback kernel against the measured FP64 add rate of this GPU
  parity       the first 10 000 reads of the batch against the oracle (mismatch counts by kind)
  c3, panel    strong-scaling legs through the sharded call (BASELINE configs[2] and [4]): FMR1 / (MGG) / DM2,
               100 002 reads, and a 50-locus x 20 000-read panel, LPT-sharded over the ranks, id-keyed NCCL gather,
               oracle sample and a sharding-independent checksum
  cpu_baseline the oracle's port of the reference's Python caller on the host cores (kind "port")
  --impl reference   the unmodified reference (byte-compiled to oracle/_ref) over a process pool on the host
               cores, as CallerWrapper.run does (kind "reference")
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree it runs from

METRIC = 'caller_reads_per_s'
UNIT = 'reads/s'
LOCUS = 'HD'
CONFIG_ID = 2


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--reads', type=int, default=100000, help='reads per GPU')
    ap.add_argument('--locus', default=LOCUS)
    ap.add_argument('--cpu-reads', type=int, default=0, help='reads of the CPU baseline sample (0 = 2 per core)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--parity-reads', type=int, default=-1,
                    help='reads of the batch checked against the oracle (-1: 10000 at N=1, 2000 at N>1)')
    ap.add_argument('--generic-only', action='store_true', help='run the catch-all DP kernel (dtw_any.cu) instead of the specialised ones')
    ap.add_argument('--mv', type=int, default=4, help='tr_calling_config.min_values_per_state')
    ap.add_argument('--no-e2e-variants', action='store_true', help='skip the int16 and raw-reads end-to-end variants')
    ap.add_argument('--raw-reads', type=int, default=25000, help='reads of the raw-reads-in end-to-end variant')
    ap.add_argument('--legs', default='c3,panel',
                    help='extra strong-scaling legs through the sharded call: c3 (FMR1, (MGG), DM2; 100k reads), '
                         'panel (C5: 50 loci x 20k reads); empty = none')
    ap.add_argument('--panel-loci', type=int, default=50)
    ap.add_argument('--panel-reads', type=int, default=20000, help='reads per locus of the panel leg')
    ap.add_argument('--c3-reads', type=int, default=33334, help='reads per locus of the c3 leg')
    ap.add_argument('--leg-base', type=int, default=2000, help='noiseless base reads per locus of a leg')
    ap.add_argument('--leg-steps', type=int, default=None, help='timed steps of each leg (default: --steps)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help="after the timed steps, write the per-read results of the last device-resident step as "
                         "DIR/<name>.npy (rank 0's batch), to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.leg_steps is None:
        args.leg_steps = args.steps
    return args


DUMP_MAX_READS = 1 << 18        # per-read arrays: every read up to this many, else a seeded sample of them
DUMP_SEQ_READS = 4096           # reads whose called sequences are written
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(path, o, n_reads):
    """The results one call_packed returned, as float64 / float32 .npy files under ``path``.

    read_index            the reads written (all of them, or a sorted sample drawn with a fixed seed)
    len1, len2, cost1, cost2, status, ttest_ties
                          per read of read_index; a read with status != 0 has no device result (NaN)
    seq_read_index        a fixed sample of read_index whose sequences are written
    seq1, seq2            those reads' called sequences (first / rescaled pass), ASCII codes, concatenated
                          in seq_read_index order; their lengths are len1 / len2 of the same reads
    """
    os.makedirs(path, exist_ok=True)
    rng = np.random.default_rng(0)
    idx = np.arange(n_reads) if n_reads <= DUMP_MAX_READS else np.sort(rng.choice(n_reads, DUMP_MAX_READS, replace=False))
    status = o['status'].cpu().numpy()[idx]
    failed = status != 0
    out = {'read_index': idx.astype(np.float64), 'status': status.astype(np.float64),
           'ttest_ties': o['ties'].cpu().numpy()[idx].astype(np.float64)}
    for k in ('len1', 'len2', 'cost1', 'cost2'):
        v = o[k].cpu().numpy()[idx].astype(np.float64)
        v[failed] = np.nan
        out[k] = v
    # the sequences of a sample of the written reads, halved until everything fits the budget
    seq_idx = np.sort(rng.choice(len(idx), min(DUMP_SEQ_READS, len(idx)), replace=False))
    seq_idx = seq_idx[~failed[seq_idx]]
    soff = np.asarray(o['seq_off'])[idx]
    seq1, seq2 = o['seq1'].cpu().numpy(), o['seq2'].cpu().numpy()
    while True:
        for k, s in (('seq1', seq1), ('seq2', seq2)):
            n = out['len' + k[-1]][seq_idx].astype(np.int64)
            out[k] = np.concatenate([s[a:a + m] for a, m in zip(soff[seq_idx], n)] or [np.zeros(0, np.uint8)]
                                    ).astype(np.float32)
        if sum(v.nbytes for v in out.values()) + 8 * len(seq_idx) <= DUMP_MAX_BYTES or len(seq_idx) <= 1:
            break
        seq_idx = seq_idx[::2]
    out['seq_read_index'] = idx[seq_idx].astype(np.float64)
    for k, v in out.items():
        np.save(os.path.join(path, k + '.npy'), v)


# ---------------------------------------------------------------------------------------------------
# CPU side (bench.py may execute oracle/ only here)
#   kind "reference": the unmodified reference's warpstr_call_sequential (src/caller/wrapper.py:292-331),
#       byte-compiled into oracle/_ref by oracle/build_ref.py, reads spread over a process pool exactly like
#       CallerWrapper.run (wrapper.py:107-109) -- what `--impl reference` times;
#   kind "port": the oracle's cell-by-cell Python port of the same DP + numpy/scipy mid-stage (4-9x faster than
#       the reference) -- the cpu_baseline of our own arm, and the fallback when oracle/_ref was not built.
# ---------------------------------------------------------------------------------------------------
_CPU_CTX = {}


def _cpu_init(locus_name, seed, kind):
    from warpstr_b200 import synth
    locus = synth.make_locus(locus_name, seed=seed)
    _CPU_CTX['kind'] = kind
    _CPU_CTX['F'] = locus.flank_length
    if kind == 'reference':
        from oracle import refshim
        ref = refshim.load()
        _CPU_CTX['ref'] = ref
        _CPU_CTX['sta'] = [ref.StateAutomata(locus.template_regex), ref.StateAutomata(locus.reverse_regex)]
        return
    from oracle import caller_oracle as co
    from warpstr_b200.automata import StateAutomata
    _CPU_CTX['tb'] = [co.tables_from(StateAutomata(locus.template_regex)),
                      co.tables_from(StateAutomata(locus.reverse_regex))]
    _CPU_CTX['co'] = co


def _cpu_one(job):
    sig, rev = job
    if _CPU_CTX['kind'] == 'reference':
        ref = _CPU_CTX['ref']
        rs = ref.wrapper.ReadSignal(name='bench', reverse=bool(rev), signal=sig)
        r = ref.wrapper.warpstr_call_sequential(rs, _CPU_CTX['F'], _CPU_CTX['sta'][int(rev)], None)
        return len(r.resc_seq)
    co = _CPU_CTX['co']
    r = co.run_read(sig, _CPU_CTX['tb'][int(rev)], _CPU_CTX['F'], bool(rev), impl='scalar')
    return len(r.resc_seq)


class CpuPool:
    """A process pool over reads, as CallerWrapper.run uses (src/caller/wrapper.py:107-109)."""

    def __init__(self, locus_name, seed, cores, kind):
        import multiprocessing as mp
        self.cores = cores
        self.pool = mp.get_context('fork').Pool(cores, initializer=_cpu_init, initargs=(locus_name, seed, kind))

    def run(self, signals, revs):
        """(seconds, allele lengths) of one pass over the sample."""
        jobs = list(zip(signals, revs))
        t0 = time.perf_counter()
        out = self.pool.map(_cpu_one, jobs, chunksize=1)
        return time.perf_counter() - t0, out

    def close(self):
        self.pool.close()
        self.pool.join()


def cpu_kind():
    from oracle import refshim
    return 'reference' if refshim.compiled_available() or refshim.source_available() else 'port'


CPU_SAMPLE_NOTE = {
    'reference': 'the unmodified reference (src/caller/wrapper.py warpstr_call_sequential, byte-compiled to oracle/_ref), '
                 'Pool over reads as CallerWrapper.run does',
    'port': "the oracle's pure-Python float64 port of caller.py:198-301 + numpy/scipy mid-stage (4-9x faster per read "
            'than the unmodified reference), Pool over reads',
}


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
             'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
             'clocks_event_reasons.sw_power_cap')
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={q}', '--format=csv,noheader,nounits',
                                          '-i', str(self.index), '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for row in self.rows:
            parts = [p.strip() for p in row.split(',')]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(names, parts[3:7]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
        return {'sm_mhz': float(np.median(sm)), 'sm_max_mhz': float(max(mx)), 'reasons': sorted(reasons),
                'samples': len(sm)}


# ---------------------------------------------------------------------------------------------------
# Strong-scaling legs (BASELINE configs[2] and [4]): a fixed multi-locus panel sharded over the ranks by DP
# cells (LPT), every rank calls its shard, one id-keyed NCCL gather returns everybody's per-read results.
# ---------------------------------------------------------------------------------------------------
LEG_SPECS = {
    'c3': dict(patterns=('FMR1', 'FMR1_MGG', 'DM2'), n_loci=3, seed=31,
               what='C3: FMR1 ((CGG){AGG}), ambiguous-base (MGG) and DM2 (in-degree 4), BASELINE configs[2]'),
    'panel': dict(patterns=None, n_loci=None, seed=51,
                  what='C5: multi-locus panel, mixed patterns with random flanks, BASELINE configs[4]'),
}


def leg_prepare(name, args, workers):
    """Host part of a leg, before CUDA exists in this process: loci and their noiseless base reads."""
    from warpstr_b200 import synth
    spec = LEG_SPECS[name]
    n_loci = spec['n_loci'] or args.panel_loci
    per = args.c3_reads if name == 'c3' else args.panel_reads
    loci = synth.make_panel(n_loci, seed=spec['seed'], patterns=spec['patterns'] or synth.PANEL_MIX)
    base = synth.make_panel_base(loci, min(args.leg_base, per), seed=spec['seed'], workers=workers)
    return dict(name=name, loci=loci, base=base, per=per, seed=spec['seed'], what=spec['what'])


def leg_run(leg, args, rank, world, barrier):
    import torch
    import torch.distributed as dist
    from warpstr_b200 import shard, synth
    from warpstr_b200.automata import StateAutomata
    from warpstr_b200.caller import CallerEngine
    loci, base, per = leg['loci'], leg['base'], leg['per']
    n_total = len(loci) * per
    regexes = []
    for loc in loci:
        regexes += [loc.template_regex, loc.reverse_regex]
    stas = [StateAutomata(rx) for rx in regexes]
    eng = CallerEngine()
    ids = np.array([eng.add_automaton(s, 110) for s in stas], dtype=np.int32)
    shapes = sorted({(i['chain_slots'], i['generic_slots']) for i in (a.info() for a in eng.automata)})
    n_states = np.array([s.n_states for s in stas], dtype=np.int64)
    locus_of, bidx, lengths_all, rev_all, truth_all = synth.panel_read_table(base, per)
    aut_all = ids[2 * locus_of + rev_all]
    shards = shard.partition_reads(lengths_all.astype(np.float64) * n_states[2 * locus_of + rev_all], world)
    counts = [len(x) for x in shards]
    mine = shards[rank]
    dev = torch.device('cuda', torch.cuda.current_device())
    d_sig, off, lengths = synth.materialize_panel_reads(base, per, mine, 0.15, leg['seed'], dev)
    aut, rev = aut_all[mine], rev_all[mine]
    d_ids = torch.as_tensor(mine, device=dev)
    # oracle sample: reads spread over every locus (and so over every rank's shard), materialised here as well
    n_sample = max(200, 4 * len(loci))
    sample = np.unique(np.linspace(0, n_total - 1, n_sample).astype(np.int64))
    want = None
    if rank == 0:
        from oracle import bulk
        s_sig, s_off, s_len = synth.materialize_panel_reads(base, per, sample, 0.15, leg['seed'], dev)
        s_host = s_sig.cpu().numpy()
        want = bulk.run_reads(regexes, 110, [s_host[o:o + n] for o, n in zip(s_off, s_len)],
                              (2 * locus_of + rev_all)[sample], rev_all[sample], workers=1)
        del s_sig

    def step():
        return shard.call_sharded_packed(eng, mine, d_sig, off, lengths, aut, rev, counts, n_total, d_ids=d_ids)

    for _ in range(max(3, args.warmup if args.warmup < 4 else 3)):
        g = step()
    barrier()
    from warpstr_b200 import _lib
    _lib.profile_enable(True)
    _lib.profile_read()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_host = time.perf_counter()
    e0.record()
    for _ in range(args.leg_steps):
        g = step()
    e1.record()
    t_host = time.perf_counter() - t_host
    barrier()
    prof = _lib.profile_read()
    _lib.profile_enable(False)
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0]) / args.leg_steps
    len1, len2, status = g['len1'].cpu().numpy(), g['len2'].cpu().numpy(), g['status'].cpu().numpy()
    cost2 = g['cost2'].cpu().numpy()
    out = None
    if rank == 0:
        ok = status == 0
        mism = 0
        for i, w in zip(sample, want):
            if w[0] == 'error':
                mism += int(status[i] == 0)
            else:
                mism += int(status[i] != 0 or len1[i] != len(w[0]) or len2[i] != len(w[1]) or cost2[i] != w[3])
        checksum = int((np.arange(1, n_total + 1, dtype=np.int64) * np.where(ok, len2, -1).astype(np.int64)).sum() % 2305843009213693951)
        loads = np.array([float((lengths_all[x].astype(np.float64) * n_states[(2 * locus_of + rev_all)[x]]).sum())
                          for x in shards])
        out = {'workload': leg['what'], 'loci': len(loci), 'automata_resident': len(stas), 'kernel_shapes': shapes,
               'reads': n_total, 'reads_per_locus': per,
               'distinct_base_reads_per_locus': int(len(base[0][2])),
               'scaling': 'strong', 'value': n_total / (ms * 1e-3), 'unit': UNIT, 'ms_per_step': ms,
               'steps': args.leg_steps,
               'path': 'shard.partition_reads (LPT by T*S) -> CallerEngine.call_packed per rank -> shard.gather_by_id '
                       '(id-keyed NCCL all_gather, 32 B/read)',
               'shard_reads': counts, 'shard_load_imbalance': float(loads.max() / loads.mean()),
               'rank0_kernel_ms_per_step': {k: prof[k]['ms'] / args.leg_steps for k in ('dp_fill_traceback', 'midstage', 'plan_upload')},
               'rank0_launches_per_step': {k: prof[k]['launches'] / args.leg_steps for k in ('dp_fill_traceback', 'midstage')},
               'rank0_host_enqueue_ms_per_step': 1e3 * t_host / args.leg_steps,
               'parity': {'oracle_sample_reads': int(len(sample)), 'oracle_mismatches': int(mism),
                          'reads_with_status': int((~ok).sum()),
                          'reads_exact_vs_truth': float(np.mean(len2[ok] == truth_all[ok])) if ok.any() else 0.0,
                          'gathered_everything': bool((status >= 0).all()),
                          'len2_checksum': checksum,
                          'len2_checksum_note': 'sum((id+1)*len2) mod 2^61-1 over all reads: identical at every N '
                                                'because the reads do not depend on the sharding'}}
    del d_sig, eng
    torch.cuda.empty_cache()
    return out


def main():
    args = parse()
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    cores = host_cores()
    config = {'workload': f'synthetic {args.locus} locus, {args.reads} reads per GPU, ~3.3k float64 samples/read, '
                          '50% reverse strand (BASELINE configs[1])',
              'reads_per_gpu': args.reads, 'locus': args.locus, 'flank_length': 110,
              'cache_policy': 'inputs (2.6 GB/GPU) and direction codes (14 GB/GPU per pass) far exceed the 126 MB L2; no flush needed',
              'parallelism': f'reads sharded over {args.gpus} GPU(s), no data-path collective; per-read results '
                             'all_gathered (NCCL) once per step when N > 1'}

    # ------------------------------------------------------------------ reference arm
    if args.impl == 'reference':
        if rank != 0:
            return
        from warpstr_b200 import synth
        kind = cpu_kind()
        n = args.cpu_reads or cores                      # one read per core and step: 5-10 s of the reference per step
        locus = synth.make_locus(args.locus, seed=1)
        reads = synth.make_reads(locus, n, seed=1000 * CONFIG_ID)
        sigs, revs = [r.signal for r in reads], [r.reverse for r in reads]
        pool = CpuPool(args.locus, 1, cores, kind)
        for _ in range(args.warmup):
            pool.run(sigs, revs)
        total = 0.0
        for _ in range(args.steps):
            dt, _ = pool.run(sigs, revs)
            total += dt
        pool.close()
        value = n * args.steps / total
        line = {'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus,
                'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * total / args.steps,
                'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64',
                'data': 'synthetic', 'config': config,
                'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': cores, 'kind': kind,
                                 'sample': f'{n} reads of the same workload per step; ' + CPU_SAMPLE_NOTE[kind]},
                'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
        print(json.dumps(line))
        return

    # ------------------------------------------------------------------ our arm
    import torch
    import torch.distributed as dist
    from warpstr_b200 import _lib, synth
    from warpstr_b200.automata import StateAutomata
    from warpstr_b200.caller import CallerEngine

    # ---- host-side preparation, before CUDA exists in this process (the process pools below fork) ----------
    locus = synth.make_locus(args.locus, seed=1)
    stas = [StateAutomata(locus.template_regex), StateAutomata(locus.reverse_regex)]
    sig, off, lengths, rev, truth = synth.make_read_batch(locus, args.reads, seed=1000 * CONFIG_ID + rank)
    n_states = np.array([stas[0].n_states, stas[1].n_states])
    n_edges = np.array([stas[0].n_edges, stas[1].n_edges])

    # the oracle over the first reads of the batch (rank 0): compared with the GPU's results further down
    n_parity = args.parity_reads if args.parity_reads >= 0 else (10000 if world == 1 else 2000)
    n_parity = min(n_parity, args.reads)
    parity_want = None
    if rank == 0 and n_parity > 0:
        from oracle import bulk
        parity_want = bulk.run_reads([locus.template_regex, locus.reverse_regex], locus.flank_length,
                                     [sig[o:o + n] for o, n in zip(off[:n_parity], lengths[:n_parity])],
                                     rev[:n_parity].astype(int), rev[:n_parity].astype(bool), workers=cores,
                                     knobs=(args.mv, 6, False, 0.5, 0.5, 'mean'))

    # CPU baseline (rank 0, single-GPU runs only)
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        n_cpu = args.cpu_reads or 2 * cores
        sample = synth.make_reads(locus, n_cpu, seed=1000 * CONFIG_ID)
        pool = CpuPool(args.locus, 1, cores, 'port')
        pool.run([r.signal for r in sample[:cores]], [r.reverse for r in sample[:cores]])   # warm the workers
        dt, cpu_len = pool.run([r.signal for r in sample], [r.reverse for r in sample])
        pool.close()
        cells = float(sum(2 * len(r.signal) * n_states[int(r.reverse)] for r in sample))
        cpu_baseline = {'value': n_cpu / dt, 'unit': UNIT, 'cores': cores, 'kind': 'port',
                        'mcups': cells / dt / 1e6,
                        'sample': f'{n_cpu} reads of the same workload; ' + CPU_SAMPLE_NOTE['port'] +
                                  ' (`--impl reference` times the unmodified reference itself)'}

    legs = [leg_prepare(name, args, max(1, min(8, cores // max(world, 1))))
            for name in args.legs.split(',') if name in LEG_SPECS]

    # ---- device ---------------------------------------------------------------------------------------------
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    from warpstr_b200.config import CallerConfig
    eng = CallerEngine(CallerConfig(min_values_per_state=args.mv))
    _lib.set_generic_only(args.generic_only)
    ids = [eng.add_automaton(s, locus.flank_length) for s in stas]
    _lib.set_generic_only(False)
    aut = np.where(rev > 0, ids[1], ids[0]).astype(np.int32)
    host = torch.from_numpy(sig).pin_memory()
    cells_pass = float((lengths.astype(np.int64) * n_states[rev.astype(np.int64)]).sum())
    alg_ops_pass = float((lengths.astype(np.int64) *
                          (4 * n_states[rev.astype(np.int64)] + 5 * n_edges[rev.astype(np.int64)])).sum())

    d_sig = host.cuda(non_blocking=True)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    from warpstr_b200 import shard

    def step_resident():
        o = eng.call_packed(d_sig, off, lengths, aut, rev, want_seq=True)
        if world > 1:   # the only exchange of the path: everybody's per-read lengths / costs / status
            o['gathered'] = shard.gather_device(o['len1'], o['len2'], o['status'], o['cost1'], o['cost2'])
        return o

    def step_e2e():
        res = eng.call_arrays(host, off, lengths, aut, rev)
        if world > 1:
            ints = torch.from_numpy(np.stack((res['len1'], res['len2'], res['status']), axis=1)).cuda()
            flts = torch.from_numpy(np.stack((res['cost1'], res['cost2']), axis=1)).cuda()
            g = shard.gather_device(ints[:, 0], ints[:, 1], ints[:, 2], flts[:, 0], flts[:, 1])
            res['gathered_len2'] = g['len2'].cpu().numpy()
        return res

    # parity of the benchmark batch itself: its first n_parity reads against the oracle (rank 0)
    o = step_resident()
    torch.cuda.synchronize()
    status = o['status'].cpu().numpy()
    len1 = o['len1'].cpu().numpy()
    len2 = o['len2'].cpu().numpy()
    cost1, cost2 = o['cost1'].cpu().numpy(), o['cost2'].cpu().numpy()
    ties = o['ties'].cpu().numpy()
    n_fallback = int((status != 0).sum())
    parity = {'reads_exact_vs_truth': float(np.mean(len2[status == 0] == truth[status == 0])) if (status == 0).any() else 0.0,
              'reads_with_status': n_fallback, 'host_fallback_reads': n_fallback + int((ties > 0).sum()),
              'ttest_tie_reads': int((ties > 0).sum()),
              'ttest_tie_note': 'reads with a t-test decision within 16 ulp of flipping (d_ttest_ties): the only reads '
                                "whose bad-repeat mask can depend on the host libm's pow rounding"}
    if parity_want is not None:
        seq1, seq2, soff = o['seq1'].cpu().numpy(), o['seq2'].cpu().numpy(), o['seq_off']
        mism = {'len': 0, 'seq': 0, 'cost': 0, 'status': 0}
        for r, w in enumerate(parity_want):
            if w[0] == 'error':
                mism['status'] += int(status[r] == 0)
                continue
            if status[r] != 0:
                mism['status'] += 1
                continue
            if ties[r] > 0:
                continue
            a = int(soff[r])
            mism['len'] += int(len1[r] != len(w[0]) or len2[r] != len(w[1]))
            mism['seq'] += int(seq1[a:a + len1[r]].tobytes().decode() != w[0] or seq2[a:a + len2[r]].tobytes().decode() != w[1])
            mism['cost'] += int(cost1[r] != w[2] or cost2[r] != w[3])
        parity['oracle_reads'] = len(parity_want)
        parity['oracle_mismatches'] = mism
        parity['oracle_note'] = ('every one of these reads through the oracle (DP in C, numpy/scipy mid-stage, Pool on the '
                                 'host cores): allele lengths, sequences and both state-wise costs compared bit for bit')
        assert not any(mism.values()), f'benchmark batch disagrees with the oracle: {mism}'
        del seq1, seq2

    fp64_rate = _lib.measure_fp64_add_rate()

    # ---- device-resident timing ------------------------------------------------------------------
    for _ in range(args.warmup):
        step_resident()
    barrier()
    gc.collect()
    gc.disable()          # no collector pauses inside the timed regions
    _lib.profile_enable(True)
    _lib.profile_read()
    sampler = ClockSampler(local_rank)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        last = None                 # each step's results are freed before the next, as when nobody keeps them
        last = step_resident()
    e1.record()
    barrier()
    clocks = sampler.stop()
    ms_total = e0.elapsed_time(e1)
    prof = _lib.profile_read()
    _lib.profile_enable(False)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last, args.reads)
    del last

    # ---- end-to-end timing (host buffers in, host arrays out) --------------------------------------
    for _ in range(args.warmup):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    per_step = []
    for _ in range(args.steps):
        ts = time.perf_counter()
        res = step_e2e()
        per_step.append(round(1e3 * (time.perf_counter() - ts), 1))
    e3.record()
    barrier()
    ms_e2e = max(e2.elapsed_time(e3), 1e3 * (time.perf_counter() - t0))
    h2d = int(host.numel() * 8)
    d2h = int(sum(v.nbytes for k, v in res.items() if not k.startswith('gathered')))

    # ---- the same batch handed over as int16 (a quarter of the bytes), and the raw-reads-in chain -----------
    def gather_host(res):
        if world > 1:
            ints = torch.from_numpy(np.stack((res['len1'], res['len2'], res['status']), axis=1)).cuda()
            flts = torch.from_numpy(np.stack((res['cost1'], res['cost2']), axis=1)).cuda()
            shard.gather_device(ints[:, 0], ints[:, 1], ints[:, 2], flts[:, 0], flts[:, 1])

    def time_e2e(fn):
        for _ in range(args.warmup):
            fn()
        barrier()
        t0 = time.perf_counter()
        ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ea.record()
        for _ in range(args.steps):
            out = fn()
        eb.record()
        barrier()
        return max(ea.elapsed_time(eb), 1e3 * (time.perf_counter() - t0)), out

    variants = {}
    if not args.no_e2e_variants:
        # (a) int16 window samples + {shift, scale}: the SURVEY 8d map norm -> DAC counts, made on the GPU
        Q_SHIFT, Q_SCALE = 90.8717 * 5.85, 9.8354 * 5.85
        len_t = torch.from_numpy(lengths.astype(np.int64)).cuda()
        first = torch.cumsum(len_t, 0) - len_t
        rep = torch.repeat_interleave(torch.arange(len(lengths), device='cuda'), len_t)
        tpos = torch.arange(int(len_t.sum().item()), device='cuda') - first[rep]
        src = torch.from_numpy(off).cuda()[rep] + tpos
        raw_off = np.zeros(len(lengths), dtype=np.int64)
        raw_off[1:] = np.cumsum((lengths[:-1].astype(np.int64) + 7) & ~7)
        dst = torch.from_numpy(raw_off).cuda()[rep] + tpos
        counts16 = torch.round(d_sig[src] * Q_SCALE + Q_SHIFT)
        d_raw16 = torch.zeros(int(raw_off[-1] + ((int(lengths[-1]) + 7) & ~7)), dtype=torch.int16, device='cuda')
        d_raw16[dst] = counts16.to(torch.int16)
        host16 = torch.empty(d_raw16.numel(), dtype=torch.int16).pin_memory()
        host16.copy_(d_raw16)
        host_ss = torch.tensor([[Q_SHIFT, Q_SCALE]] * len(lengths), dtype=torch.float64).pin_memory()
        # the float64 windows those samples stand for, for the check: the reference's (data - shift) / scale
        d_q64 = torch.zeros_like(d_sig)
        # (a tensor divisor: torch turns division by a Python scalar into a multiplication by its reciprocal)
        d_q64[src] = (counts16 - Q_SHIFT) / torch.full_like(counts16, Q_SCALE)
        want16 = eng.call_packed(d_q64, off, lengths, aut, rev, want_seq=False)
        want16 = {k: want16[k].cpu().numpy() for k in ('len1', 'len2', 'cost1', 'cost2', 'status')}
        q_sample = [d_q64[int(off[r]):int(off[r]) + int(lengths[r])].cpu().numpy() for r in range(0, len(lengths), max(1, len(lengths) // 48))][:48]
        del d_raw16, d_q64, src, dst, rep, tpos, counts16

        def step_i16():
            res = eng.call_arrays_quantized(host16, raw_off, lengths, host_ss, aut, rev)
            gather_host(res)
            return res

        ms_i16, r16 = time_e2e(step_i16)
        same = all(np.array_equal(r16[k], want16[k], equal_nan=True) for k in want16)
        variants['e2e_int16'] = {
            'ms': ms_i16, 'h2d': int(host16.numel() * 2 + host_ss.numel() * 8),
            'd2h': int(sum(v.nbytes for v in r16.values() if isinstance(v, np.ndarray))),
            'api': 'CallerEngine.call_arrays_quantized (pinned int16 window samples + {shift, scale} per read -> '
                   'wstr_dequantize_batch -> wstr_call_batch -> host arrays)',
            'workload': 'the same reads in DAC counts, raw = rint((90.8717 + 9.8354 x) 5.85) (SURVEY 8d); the device '
                        "re-creates the float64 windows with the reference's (data - shift) / scale",
            'parity': {'all_reads_equal_the_float64_call_on_the_same_windows': bool(same)}}
        if rank == 0:
            from oracle import caller_oracle as co
            tbs = [co.tables_from(s_) for s_ in stas]
            mism = 0
            for k, x in enumerate(q_sample):
                r = k * max(1, len(lengths) // 48)
                w = co.run_read(x, tbs[int(rev[r])], locus.flank_length, bool(rev[r]), impl='c', bulk=True)
                mism += int(r16['len2'][r] != len(w.resc_seq) or r16['cost2'][r] != w.resc_cost or r16['len1'][r] != len(w.seq))
            variants['e2e_int16']['parity'].update(oracle_reads=len(q_sample), oracle_mismatches=mism)
        assert same, 'int16 ingestion disagrees with the float64 call on the same windows'
        del host16, r16

        # (b) raw reads in: whole int16 reads (window + 8192 flank-like samples, spikes at 1e-4) -> normalisation
        # kernel -> caller, windows never on the host.  A quarter of the batch (the generator is the slow part).
        n_raw = max(1, min(len(lengths), args.raw_reads))
        PAD = 8192
        gen = torch.Generator(device='cuda')
        gen.manual_seed(1000 * CONFIG_ID + 77 + rank)
        ln = torch.from_numpy(lengths[:n_raw].astype(np.int64)).cuda()
        full_len = ln + PAD
        roff = np.zeros(n_raw + 1, dtype=np.int64)
        roff[1:] = np.cumsum(lengths[:n_raw].astype(np.int64) + PAD)
        total_raw = int(roff[-1])
        from warpstr_b200.pore_model import get_pore_model
        table = torch.from_numpy(np.ascontiguousarray(get_pore_model().table)).cuda()
        kidx = torch.randint(0, table.numel(), (total_raw // 9 + 2,), generator=gen, device='cuda')
        full = torch.repeat_interleave(table[kidx], 9)[:total_raw] + 0.15 * torch.randn(total_raw, generator=gen, dtype=torch.float64, device='cuda')
        rep = torch.repeat_interleave(torch.arange(n_raw, device='cuda'), ln)
        tpos = torch.arange(int(ln.sum().item()), device='cuda') - (torch.cumsum(ln, 0) - ln)[rep]
        full[torch.from_numpy(roff[:-1]).cuda()[rep] + PAD // 2 + tpos] = d_sig[torch.from_numpy(off[:n_raw]).cuda()[rep] + tpos]
        counts = torch.round((90.8717 + 9.8354 * full) * 5.85)
        spikes = torch.rand(total_raw, generator=gen, device='cuda') < 1e-4
        counts = torch.where(spikes, torch.where(torch.rand(total_raw, generator=gen, device='cuda') < 0.5, 1500.0, 100.0), counts)
        host_raw = torch.empty(total_raw, dtype=torch.int16).pin_memory()
        host_raw.copy_(counts.to(torch.int16))
        win_lo = np.full(n_raw, PAD // 2, dtype=np.int32)
        win_hi = (win_lo + lengths[:n_raw] - 1).astype(np.int32)
        del full, counts, spikes, rep, tpos, kidx

        def step_raw():
            res = eng.call_arrays_raw(host_raw, roff, win_lo, win_hi, aut[:n_raw], rev[:n_raw], 'Brute')
            gather_host(res)
            return res

        ms_raw, rr = time_e2e(step_raw)
        variants['e2e_raw'] = {
            'ms': ms_raw, 'reads': n_raw, 'h2d': int(total_raw * 2),
            'd2h': int(sum(v.nbytes for v in rr.values() if isinstance(v, np.ndarray))),
            'api': 'CallerEngine.call_arrays_raw (pinned int16 whole reads + windows -> wstr_normalize_batch (Brute spike '
                   'removal, MAD normalisation, slice) -> wstr_call_batch -> host arrays); the get_workload -> '
                   'CallerWrapper.run chain of src/caller/wrapper.py:44-54,104-120, windows never on the host',
            'workload': f'{n_raw} reads of the batch, each embedded in a raw read of T + {PAD} samples (flank-like '
                        'filler, spikes at 1e-4), SURVEY 8d'}
        if rank == 0:
            from oracle import caller_oracle as co
            from oracle import normalize_oracle as no
            tbs = [co.tables_from(s_) for s_ in stas]
            mism, checked = 0, 0
            for r in range(0, n_raw, max(1, n_raw // 32)):
                raw = host_raw.numpy()[roff[r]:roff[r + 1]]
                x = no.get_data_processed(raw, (int(win_lo[r]), int(win_hi[r])), 'Brute')
                w = co.run_read(x, tbs[int(rev[r])], locus.flank_length, bool(rev[r]), impl='c', bulk=True)
                mism += int(rr['status'][r] != 0 or rr['len2'][r] != len(w.resc_seq) or rr['cost2'][r] != w.resc_cost)
                checked += 1
            variants['e2e_raw']['parity'] = {'oracle_reads': checked, 'oracle_mismatches': mism,
                                             'note': 'numpy normalisation + oracle call of the same raw reads'}
        del host_raw, rr

    t = torch.tensor([ms_total, ms_e2e] + [v['ms'] for v in variants.values()], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, ms_e2e = float(t[0]), float(t[1])
    for i, v in enumerate(variants.values()):
        v['ms'] = float(t[2 + i])

    # ---- strong-scaling legs through the sharded call ------------------------------------------------------
    inf = [eng.automata[i].info() for i in ids]
    del d_sig, host, o, res
    variants_keep = variants
    eng = None
    gc.collect()
    torch.cuda.empty_cache()
    leg_out = {}
    for leg in legs:
        leg_out[leg['name']] = leg_run(leg, args, rank, world, barrier)

    if rank == 0:
        total_reads = args.reads * world
        fill = prof['dp_fill_traceback']
        mid = prof['midstage']
        fill_ms_launch = fill['ms'] / max(fill['launches'], 1)
        # a launch covers one pass over this rank's batch (single wave) -> algorithmic ops per launch
        waves = max(1, fill['launches'] // (2 * args.steps))
        ops_per_launch = alg_ops_pass / waves
        achieved = ops_per_launch / (fill_ms_launch * 1e-3) / 1e12
        gcups = cells_pass / waves / (fill_ms_launch * 1e-3) / 1e9
        traffic = None
        tpath = os.path.join(ROOT, 'profiles', 'fill_traffic.json')
        if os.path.exists(tpath):
            try:
                tj = json.load(open(tpath))
                traffic = tj.get('dram_bytes_per_launch_at_bench_size') * (args.reads / waves) / tj.get('reads', 100000)
            except Exception:
                traffic = None
        # FP64-pipe instructions the kernel executes per DP row of one read: per lane 5 DADD per chain slot,
        # 4 + candidates per generic slot, one DSETP per candidate = 4 K + 2 NB (K slots per lane, NB = direction
        # bits per lane and row = candidates), times 32 lanes
        fp64_per_row = float(np.mean([32 * (4 * a['states_per_lane'] + 2 * a['dir_bits_per_row']) for a in inf]))
        rows_pass = float(lengths.astype(np.int64).sum())
        secs = fill_ms_launch * 1e-3
        hbm_peak = None
        ppath = os.path.join(ROOT, 'MEASURED_PEAKS.json')
        if os.path.exists(ppath):
            try:
                hbm_peak = float(json.load(open(ppath))['hbm_gbs'])
            except Exception:
                hbm_peak = None
        hbm_src = 'MEASURED_PEAKS.json hbm_gbs (measured)' if hbm_peak else 'fallback 6650 GB/s (B200_PROFILING.md)'
        hbm_peak = hbm_peak or 6650.0
        # algorithmic HBM bytes of one pass: direction codes written once and read once by the traceback
        # (128 B per 3 rows), signal read (8 B/row), trace written (4 B/row)
        alg_bytes = rows_pass / waves * (2 * 128.0 / 3.0 + 8.0 + 4.0)
        line = {
            'metric': METRIC, 'value': total_reads * args.steps / (ms_total * 1e-3), 'unit': UNIT,
            'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms_total / args.steps,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': config,
            'dp_gcups': gcups * world,
            'dp_gcups_note': 'cells (T*S per pass) / device time of the fill+traceback kernel, all GPUs',
            'e2e_float64': {'value': total_reads * args.steps / (ms_e2e * 1e-3), 'unit': UNIT,
                            'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                            'api': 'CallerEngine.call_arrays (pinned host float64 windows, the type of the reference\'s '
                                   'ReadSignal.signal -> wstr_call_batch -> host arrays)',
                            'ms_each_step': per_step},
            # this library's kernels inside the timed region: per fill launch one zero_kernel (its wave's work
            # counters); per call 5 mid-stage kernels (3 after the first pass, 2 after the second), their 2
            # zero_kernels and the upload_kernel of the host plan
            'gpu_launches': int(2 * fill['launches'] + 3 * (mid['launches'] // 2) + 2 * (mid['launches'] - mid['launches'] // 2)
                                + 3 * args.steps),
            'kernel_ms_per_step': {'dp_fill_traceback': fill['ms'] / args.steps, 'midstage': mid['ms'] / args.steps},
            'roofline': {'bound': 'fp64_add_pipe', 'achieved': achieved, 'peak': fp64_rate, 'unit': 'T FP64 add-class op/s',
                         'frac': achieved / fp64_rate, 'traffic': traffic,
                         'kernel': 'dtw_fill_kernel (fill + traceback)',
                         'note': 'the DP is FP64 add/compare work, not HBM- or tensor-bound (SURVEY 8d); achieved = '
                                 'algorithmic ops (4 + 5 E/S per cell) per launch / launch time; frac_executed counts '
                                 'the FP64-pipe instructions the kernel really issues',
                         'peak_source': 'measured in this run by wstr_measure_fp64_add_rate (DADD stream on all SMs); '
                                        'MEASURED_PEAKS.json has no FP64 figure',
                         'algorithmic_ops_per_cell': alg_ops_pass / cells_pass,
                         'executed_fp64_instr_per_row': fp64_per_row,
                         'frac_executed': rows_pass / waves * fp64_per_row / secs / 1e12 / fp64_rate,
                         'hbm': {'bound': 'hbm', 'achieved': alg_bytes / secs / 1e9, 'peak': hbm_peak, 'unit': 'GB/s',
                                 'frac': alg_bytes / secs / 1e9 / hbm_peak, 'peak_source': hbm_src,
                                 'algorithmic_bytes_per_launch': alg_bytes}},
            'cpu_baseline': cpu_baseline,
            'clocks': clocks,
            'parity': parity,
        }
        for name, v in variants.items():
            n_v = v.get('reads', args.reads) * world
            line[name] = {'value': n_v * args.steps / (v['ms'] * 1e-3), 'unit': UNIT, 'reads_per_gpu': v.get('reads', args.reads),
                          'h2d_bytes_per_step': v['h2d'], 'd2h_bytes_per_step': v['d2h'], 'api': v['api'],
                          'workload': v['workload'], 'parity': v.get('parity')}
        # The headline end-to-end figure: the batch handed over as what the reads are on disk and what determines
        # the float64 windows bit for bit -- int16 samples + {shift, scale} per read, a quarter of the bytes over
        # PCIe (with eight GPUs on one host the float64 form is bound by the host's memory system, see
        # e2e_float64).  Without the variants (--no-e2e-variants) the float64 form stands in.
        if 'e2e_int16' in line:
            line['e2e'] = dict(line.pop('e2e_int16'), form='int16 window samples + {shift, scale} (e2e_float64: the same '
                                                            'call on float64 windows; e2e_raw: whole raw reads in)')
        else:
            line['e2e'] = dict(line['e2e_float64'], form='float64 windows (int16 variants skipped)')
        line.update({k: v for k, v in leg_out.items() if v is not None})
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
