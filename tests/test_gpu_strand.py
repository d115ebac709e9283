"""GPU: reads without a strand (DESIGN.md section 4.5).  Such a read is searched with both strands' automata in
one wstr_locate_batch launch; each search matches the C oracle (oracle/locate_oracle.c) bit for bit, the strand
chosen is the true one on synthetic reads, and the calls, the bundled reads' alleles and main_wrapper's files are
those of the same reads with their strands given."""
import os

import numpy as np
import pytest

import _h5write as hw
from oracle import locate as lo_oracle
from warpstr_b200 import synth

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), 'golden')


def _filler(rng, n, pm):
    """~n samples of squiggled random sequence."""
    return synth.squiggle(rng, synth.random_flank(rng, n // 9 + 8), pm)[:n]


def _whole_reads(locus, n, seed, pad=(20_000, 200_000), noise=0.15):
    """make_reads windows embedded in squiggled random sequence: (signals, true windows, true strands)."""
    pm = synth.get_pore_model()
    rng = np.random.default_rng([seed, 0x57A])
    reads = synth.make_reads(locus, n, seed=seed, noise=noise)
    sigs, wins = [], []
    for r in reads:
        a, b = (int(x) for x in rng.integers(pad[0] // 2, pad[1] // 2 + 1, size=2))
        left, right = _filler(rng, a, pm), _filler(rng, b, pm)
        sigs.append(np.concatenate((left, r.signal, right)))
        wins.append((len(left), len(left) + len(r.signal) - 1))
    return sigs, wins, [r.reverse for r in reads]


def _engine(locus, mv=4):
    from warpstr_b200.automata import StateAutomata
    from warpstr_b200.caller import CallerEngine
    from warpstr_b200.config import CallerConfig
    stas = [StateAutomata(locus.template_regex), StateAutomata(locus.reverse_regex)]
    eng = CallerEngine(CallerConfig(min_values_per_state=mv))
    return eng, stas, [eng.add_automaton(s, locus.flank_length) for s in stas]


def _locate(eng, sigs, aut):
    from warpstr_b200.caller import pack_signals
    host, off, lengths = pack_signals(sigs)
    return eng.locate_packed(host.to(eng.device), off, lengths, aut)


def _bits(x):
    return np.asarray(x, dtype=np.float64).view(np.int64)


@pytest.mark.parametrize('name,mv', [('HD', 4), ('FMR1', 4), ('DM2', 4), ('CAN', 4), ('C9ORF72_100', 4),
                                     ('HD', 2), ('DM2', 8)])
def test_both_strands_match_oracle(built_lib, name, mv):
    """Pairs and single entries in one launch: every search of a pair and every single entry equal the oracle with
    that automaton; the chosen strand's window is the oracle's under choose_strand."""
    from warpstr_b200.caller import choose_strand
    locus = synth.make_locus(name, seed=17)
    eng, stas, ids = _engine(locus, mv)
    sigs, _, rev = _whole_reads(locus, 6, seed=19, pad=(10_000, 50_000))
    pm = synth.get_pore_model()
    sigs.append(_filler(np.random.default_rng(6), 30_000, pm))        # pure filler: found on neither strand
    sigs.append(sigs[0][:40])                                            # shorter than either strand's path
    rev += [None, None]
    aut = [tuple(ids) if k % 2 == 0 or r is None else ids[int(r)] for k, r in enumerate(rev)]
    pair = np.array([isinstance(a, tuple) for a in aut])
    got = _locate(eng, sigs, aut)
    thr = os.cpu_count() or 8
    p = np.flatnonzero(pair)
    for s in (0, 1):
        lo, hi, score, status = lo_oracle.locate_batch([sigs[r] for r in p], [stas[s]] * len(p), mv, threads=thr)
        assert np.array_equal(got['strand_status'][p, s], status), (s, got['strand_status'][p, s], status)
        assert np.array_equal(got['strand_lo'][p, s], lo) and np.array_equal(got['strand_hi'][p, s], hi), s
        assert np.array_equal(_bits(got['strand_score'][p, s]), _bits(score)), s
    strand, col, status, score = choose_strand(got['strand_status'][p], got['strand_score'][p])
    assert np.array_equal(got['strand'][p], strand) and np.array_equal(got['status'][p], status)
    assert np.array_equal(_bits(got['score'][p]), _bits(score))
    assert np.array_equal(got['lo'][p], got['strand_lo'][p, col]) and np.array_equal(got['hi'][p], got['strand_hi'][p, col])
    q = np.flatnonzero(~pair)
    lo, hi, score, status = lo_oracle.locate_batch([sigs[r] for r in q], [stas[int(rev[r])] for r in q], mv, threads=thr)
    assert np.array_equal(got['status'][q], status) and np.array_equal(_bits(got['score'][q]), _bits(score))
    assert np.array_equal(got['lo'][q], lo) and np.array_equal(got['hi'][q], hi)
    assert (got['strand'][q] == -1).all() and (got['strand_status'][q] == -1).all()
    assert np.isnan(got['strand_score'][q]).all()
    # the filler read and the short read
    assert got['strand'][6] == -1 and got['status'][6] == 1 and (got['strand_status'][6] == 1).all()
    assert got['strand'][7] == -1 and got['status'][7] == 2 and (got['strand_status'][7] == 2).all()
    if mv == 4:
        assert (got['strand'][p[:-2]] == np.array(rev)[p[:-2]].astype(int)).all()


def _strand_accuracy(noise, counts):
    """Per locus: every read searched on both strands.  Returns (reads, found, right strand, gaps), the gap being
    the wrong strand's score minus the right one's for the reads found on the right strand."""
    total = found = right = 0
    gaps = []
    for k, (name, n) in enumerate(counts):
        locus = synth.make_locus(name, seed=30 + k)
        eng, _, ids = _engine(locus)
        sigs, _, rev = _whole_reads(locus, n, seed=40 + k, pad=(4_000, 20_000), noise=noise)
        got = _locate(eng, sigs, [tuple(ids)] * n)
        truth = np.array(rev, dtype=np.int8)
        ok = got['strand'] == truth
        total += n
        found += int((got['strand'] >= 0).sum())
        right += int(ok.sum())
        sc = got['strand_score'][ok]
        t = truth[ok]
        gaps.append(sc[np.arange(len(t)), 1 - t] - sc[np.arange(len(t)), t])
        print(f'strand accuracy, noise {noise}, {name}: {int(ok.sum())} of {n} right, '
              f'{int((got["strand"] >= 0).sum())} found')
    gaps = np.concatenate(gaps)
    print(f'strand accuracy, noise {noise}: {right} of {total} right, {found} found; score gap (wrong - right) '
          f'min {gaps.min():.1f} p1 {np.percentile(gaps, 1):.1f} p50 {np.percentile(gaps, 50):.1f}')
    return total, found, right, gaps


def test_strand_accuracy_on_synthetic_truth(built_lib):
    counts = [('HD', 2000), ('FMR1', 300), ('DM2', 300), ('CAN', 300)]
    total, found, right, gaps = _strand_accuracy(0.15, counts)
    assert right == total and (gaps > 0).all()
    total, found, right, _ = _strand_accuracy(0.30, counts)
    assert found > 0 and right >= 0.99 * found


def _hd_raw_reads(n, seed):
    locus = synth.make_locus('HD', seed=seed)
    reads = synth.make_reads(locus, n, seed=seed + 1, noise=0.15)
    rng = np.random.default_rng(seed + 2)
    raws, wins = [], []
    for r in reads:
        raw, lo, hi = synth.to_raw_int16(rng, r.signal, pad=int(rng.integers(8_000, 30_000)), spike_rate=1e-4)
        raws.append(raw)
        wins.append((lo, hi))
    return locus, raws, wins, [r.reverse for r in reads]


def _wrapper(locus):
    from warpstr_b200.wrapper import CallerWrapper, Locus, flanks_from_template
    return CallerWrapper(Locus(name='LOC', sequence=locus.sequence, flank_length=locus.flank_length),
                         flanks=flanks_from_template(locus.left, locus.right))


def _same_calls(cw, run, reads, truth):
    detected = run(reads, None, [None] * len(reads))
    loc_d = dict(cw.engine.last_located)
    given = run(reads, None, truth)
    loc_g = cw.engine.last_located
    assert loc_d['strand'].tolist() == [int(t) for t in truth]
    assert (loc_d['status'] == 0).all() and (loc_g['status'] == 0).all()
    assert np.array_equal(loc_d['lo'], loc_g['lo']) and np.array_equal(loc_d['hi'], loc_g['hi'])
    for k, (a, b) in enumerate(zip(detected, given)):
        assert a == b, k


def test_calls_same_as_with_given_strands(built_lib, tmp_path):
    from warpstr_b200.fast5 import raw_chunks
    locus, raws, _, truth = _hd_raw_reads(24, seed=50)
    cw = _wrapper(locus)
    _same_calls(cw, cw.run_raw, raws, truth)
    p = str(tmp_path / 'run.fast5')
    hw.write_multi(p, {f'r{k}': r for k, r in enumerate(raws)}, 'vbz0', chunk=4000)
    reads = [raw_chunks(p, f'r{k}') for k in range(len(raws))]
    _same_calls(cw, cw.run_compressed, reads, truth)


def test_given_window_needs_a_strand(built_lib):
    from warpstr_b200.wrapper import ReadSignal
    locus, raws, wins, truth = _hd_raw_reads(2, seed=55)
    cw = _wrapper(locus)
    with pytest.raises(ValueError, match='#1'):
        cw.run_raw(raws, wins, [truth[0], None])
    with pytest.raises(ValueError, match='nameless'):
        cw.run([ReadSignal('named', False, np.zeros(100)), ReadSignal('nameless', None, np.zeros(100))])


def _fixture():
    z = np.load(os.path.join(GOLD, 'c1_bundled.npz'))
    raws = [np.cumsum(z[f'raw_delta{i}'].astype(np.int64)).astype(np.int16) for i in range(len(z['names']))]
    return z, raws


def _bundled_locus(z):
    return synth.SynthLocus(name='LOC', sequence=str(z['sequence']), left=str(z['left']), right=str(z['right']),
                            units=(), flank_length=int(z['flank_length']))


def test_bundled_reads_strands_detected(built_lib):
    z, raws = _fixture()
    cw = _wrapper(_bundled_locus(z))
    loc = cw.locate_raw(raws, [None] * len(raws))
    assert (loc['status'] == 0).all()
    assert loc['strand'].tolist() == [int(bool(r)) for r in z['reverse']]
    res = cw.run_raw(raws, None, [None] * len(raws))
    assert [len(r.seq) for r in res] == z['len1'].tolist()
    assert [len(r.resc_seq) for r in res] == z['len2'].tolist()
    assert sorted(set(len(r.resc_seq) for r in res)) == [40, 44]


OUT_FILES = ('overview.csv', 'predictions/sequences/all.fasta', 'predictions/sequences/sequences_template.fasta',
             'predictions/sequences/sequences_reverse.fasta')
COMPLEX = 'predictions/complexSTR_analysis/complex_repeat_units.csv'


def _main_wrapper(tmp_path, tag, locus, rows):
    """caller_only.prepare + main_wrapper on ``rows`` (fast5 path, read name, reverse, lo, hi as CSV cells):
    (overview DataFrame, {output file: bytes})."""
    import warnings
    import pandas as pd
    from warpstr_b200 import caller_only
    from warpstr_b200.wrapper import Locus, flanks_from_template, main_wrapper
    csv_path = str(tmp_path / f'{tag}.csv')
    with open(csv_path, 'w') as fh:
        fh.write('fast5_path,locus,read_name,reverse,l_start_raw,r_end_raw\n')
        for p, n, rv, a, b in rows:
            fh.write(f'{p},LOC,{n},{rv},{a},{b}\n')
    out = str(tmp_path / f'out_{tag}')
    caller_only.prepare(out, csv_path)
    path = os.path.join(out, 'LOC')
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)      # (host mid-stage notes, if any)
        main_wrapper(Locus(name='LOC', sequence=locus.sequence, flank_length=locus.flank_length, path=path),
                     flanks=flanks_from_template(locus.left, locus.right))
    files = {}
    for f in OUT_FILES + (COMPLEX,):
        if os.path.exists(os.path.join(path, f)):
            with open(os.path.join(path, f), 'rb') as fh:
                files[f] = fh.read()
    return pd.read_csv(os.path.join(path, 'overview.csv')).set_index('read_name'), files


def test_main_wrapper_bundled_reads_without_strands(built_lib, tmp_path):
    z, raws = _fixture()
    names = [str(n) for n in z['names']]
    paths = []
    for k in range(2):
        p = str(tmp_path / f'run{k}.fast5')
        hw.write_multi(p, {n: raws[i] for i, n in enumerate(names) if i % 2 == k}, 'vbz0', chunk=4000)
        paths.append(p)
    locus = _bundled_locus(z)
    truth = [bool(r) for r in z['reverse']]
    df, files = _main_wrapper(tmp_path, 'none', locus, [(paths[i % 2], n, '', '', '') for i, n in enumerate(names)])
    df = df.loc[names]
    assert df['results'].tolist() == z['len2'].tolist() and df['orig'].tolist() == z['len1'].tolist()
    assert df['reverse'].tolist() == truth
    assert np.abs(df['l_start_raw'].to_numpy() - z['l_start_raw']).max() <= 50
    assert np.abs(df['r_end_raw'].to_numpy() - z['r_end_raw']).max() <= 50
    _, given = _main_wrapper(tmp_path, 'given', locus,
                             [(paths[i % 2], n, truth[i], '', '') for i, n in enumerate(names)])
    assert set(files) == set(OUT_FILES) and files == given


def test_main_wrapper_two_unit_locus_without_strands(built_lib, tmp_path):
    """HD has two repeat units, so the complex-unit CSV (which carries each read's strand) is written too."""
    locus, raws, _, truth = _hd_raw_reads(12, seed=60)
    p = str(tmp_path / 'run.fast5')
    hw.write_multi(p, {f'r{k}': r for k, r in enumerate(raws)}, 'vbz0', chunk=4000)
    df, files = _main_wrapper(tmp_path, 'none', locus, [(p, f'r{k}', '', '', '') for k in range(len(raws))])
    assert df['reverse'].tolist() == truth and (df['results'] > 0).all()
    _, given = _main_wrapper(tmp_path, 'given', locus, [(p, f'r{k}', truth[k], '', '') for k in range(len(raws))])
    assert set(files) == set(OUT_FILES + (COMPLEX,)) and files == given


def test_main_wrapper_mixed_rows(built_lib, tmp_path):
    """Strand and window given; strand only; neither; a filler read with neither: the filler read keeps empty
    reverse, window and result cells and is named in the one warning, the other rows are called."""
    import pandas as pd
    from warpstr_b200 import caller_only
    from warpstr_b200.wrapper import Locus, flanks_from_template, main_wrapper
    locus, raws, wins, truth = _hd_raw_reads(3, seed=70)
    rng = np.random.default_rng(71)
    filler, _, _ = synth.to_raw_int16(rng, _filler(rng, 20_000, synth.get_pore_model()), pad=2000)
    p = str(tmp_path / 'run.fast5')
    hw.write_multi(p, {'both': raws[0], 'strand': raws[1], 'neither': raws[2], 'lost': filler}, 'vbz0', chunk=4000)
    csv_path = str(tmp_path / 'reads.csv')
    with open(csv_path, 'w') as fh:
        fh.write('fast5_path,locus,read_name,reverse,l_start_raw,r_end_raw\n')
        fh.write(f'{p},LOC,both,{truth[0]},{wins[0][0]},{wins[0][1]}\n')
        fh.write(f'{p},LOC,strand,{truth[1]},,\n')
        fh.write(f'{p},LOC,neither,,,\n')
        fh.write(f'{p},LOC,lost,,,\n')
    out = str(tmp_path / 'out')
    caller_only.prepare(out, csv_path)
    loc = Locus(name='LOC', sequence=locus.sequence, flank_length=locus.flank_length, path=os.path.join(out, 'LOC'))
    with pytest.warns(RuntimeWarning, match='lost') as rec:
        main_wrapper(loc, flanks=flanks_from_template(locus.left, locus.right))
    lost_warnings = [w for w in rec if 'not found' in str(w.message)]
    assert len(lost_warnings) == 1 and 'neither' not in str(lost_warnings[0].message)
    df = pd.read_csv(os.path.join(out, 'LOC', 'overview.csv')).set_index('read_name')
    assert (df.loc[['both', 'strand', 'neither'], 'results'] > 0).all()
    assert df.loc[['both', 'strand', 'neither'], 'reverse'].tolist() == truth
    assert (df.loc['both', 'l_start_raw'], df.loc['both', 'r_end_raw']) == wins[0]
    for k, n in ((1, 'strand'), (2, 'neither')):
        assert abs(df.loc[n, 'l_start_raw'] - wins[k][0]) < 60 and abs(df.loc[n, 'r_end_raw'] - wins[k][1]) < 60
    for c in ('reverse', 'l_start_raw', 'r_end_raw', 'results', 'orig', 'dtw_cost1', 'dtw_cost2'):
        assert pd.isna(df.loc['lost', c]), c
