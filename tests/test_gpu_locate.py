"""GPU: the STR window search in whole reads (wstr_locate_batch, DESIGN.md section 4.5) against the C oracle
(oracle/locate_oracle.c) bit for bit, its accuracy on synthetic truth, and the located-then-called routes
(CallerEngine.call_raw_batch / call_vbz_batch with windows=None, main_wrapper on an overview without windows)
on the bundled reads."""
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


def _whole_reads(locus, n, seed, pad=(20_000, 200_000), noise=0.15, decoy=False):
    """make_reads windows embedded in squiggled random sequence: (signals, true windows, reverse flags,
    true STR lengths).  ``decoy``: a lone copy of the read's left flank in front of the window and of its right
    flank behind it, 2 000-8 000 samples away."""
    pm = synth.get_pore_model()
    rng = np.random.default_rng([seed, 0x10C])
    reads = synth.make_reads(locus, n, seed=seed, noise=noise)
    sigs, wins = [], []
    for r in reads:
        a, b = (int(x) for x in rng.integers(pad[0] // 2, pad[1] // 2 + 1, size=2))
        left, right = _filler(rng, a, pm), _filler(rng, b, pm)
        if decoy:
            lf, rf = (locus.left, locus.right) if not r.reverse else \
                (synth.reverse_complement(locus.right), synth.reverse_complement(locus.left))
            gap = int(rng.integers(2000, 8000))
            left = np.concatenate((left[:a - gap - 1200], synth.squiggle(rng, lf, pm, noise), left[a - gap:]))
            right = np.concatenate((right[:gap], synth.squiggle(rng, rf, pm, noise), right[gap + 1200:]))
        sigs.append(np.concatenate((left, r.signal, right)))
        wins.append((len(left), len(left) + len(r.signal) - 1))
    return sigs, wins, [r.reverse for r in reads], [r.truth_len for r in reads]


def _engine(locus, mv=4, generic=False):
    from warpstr_b200 import _lib
    from warpstr_b200.automata import StateAutomata
    from warpstr_b200.caller import CallerEngine
    from warpstr_b200.config import CallerConfig
    stas = [StateAutomata(locus.template_regex), StateAutomata(locus.reverse_regex)]
    eng = CallerEngine(CallerConfig(min_values_per_state=mv))
    _lib.set_generic_only(generic)
    try:
        ids = [eng.add_automaton(s, locus.flank_length) for s in stas]
    finally:
        _lib.set_generic_only(False)
    return eng, stas, ids


def _locate(eng, sigs, aut):
    from warpstr_b200.caller import pack_signals
    host, off, lengths = pack_signals(sigs)
    return eng.locate_packed(host.to(eng.device), off, lengths, aut)


def _same_as_oracle(got, sigs, tbs, mv):
    lo, hi, score, status = lo_oracle.locate_batch(sigs, tbs, mv, threads=os.cpu_count() or 8)
    assert np.array_equal(got['status'], status), (got['status'], status)
    assert np.array_equal(got['lo'], lo) and np.array_equal(got['hi'], hi)
    assert np.array_equal(got['score'].view(np.int64), score.view(np.int64))


@pytest.mark.parametrize('name,mv', [('HD', 4), ('FMR1', 4), ('DM2', 4), ('CAN', 4), ('C9ORF72_100', 4),
                                     ('HD', 2), ('DM2', 8), ('CAN', 2), ('FMR1', 8)])
def test_kernel_matches_oracle(built_lib, name, mv):
    locus = synth.make_locus(name, seed=7)
    eng, stas, ids = _engine(locus, mv)
    sigs, wins, rev, _ = _whole_reads(locus, 6, seed=11, pad=(20_000, 120_000))
    pm = synth.get_pore_model()
    sigs.append(_filler(np.random.default_rng(5), 30_000, pm))        # pure filler: nothing to find
    rev.append(False)
    sigs.append(sigs[0][:40])                                            # shorter than any path
    rev.append(True)
    aut = [ids[int(r)] for r in rev]
    got = _locate(eng, sigs, aut)
    _same_as_oracle(got, sigs, [stas[int(r)] for r in rev], mv)
    assert got['status'][6] == 1 and got['status'][7] == 2, got['score'][6:]
    if mv == 4:
        assert (got['status'][:6] == 0).all()


def test_catch_all_automaton_and_one_long_read(built_lib):
    """An automaton created for the catch-all caller kernel, reads up to 200 000 filler samples."""
    locus = synth.make_locus('HD', seed=8)
    eng, stas, ids = _engine(locus, 4, generic=True)
    sigs, wins, rev, _ = _whole_reads(locus, 3, seed=12, pad=(150_000, 200_000))
    aut = [ids[int(r)] for r in rev]
    got = _locate(eng, sigs, aut)
    _same_as_oracle(got, sigs, [stas[int(r)] for r in rev], 4)
    assert (got['status'] == 0).all()


def test_rings_in_the_workspace(built_lib):
    """Dwell 10 on ~1 600 states: the caller's catch-all kernel takes the automaton, the window search's rings
    (12 B per state and dwell) do not fit shared memory and live in the workspace."""
    locus = synth.make_locus('HD', seed=6, flank_length=780)
    eng, stas, ids = _engine(locus, 10)
    spad = (max(s.n_states for s in stas) + 31) // 32 * 32
    assert 12 * 10 * spad + 32 * spad + 2 * 128 * 8 > 226 * 1024     # rings + the rest of the kernel's shared memory
    sigs, wins, rev, _ = _whole_reads(locus, 3, seed=15, pad=(10_000, 20_000))
    aut = [ids[int(r)] for r in rev]
    _same_as_oracle(_locate(eng, sigs, aut), sigs, [stas[int(r)] for r in rev], 10)


def test_decoy_flanks(built_lib):
    """A lone copy of either flank elsewhere in the read does not pull the window off the full match."""
    locus = synth.make_locus('HD', seed=9)
    eng, stas, ids = _engine(locus)
    sigs, wins, rev, _ = _whole_reads(locus, 24, seed=13, pad=(20_000, 40_000), decoy=True)
    got = _locate(eng, sigs, [ids[int(r)] for r in rev])
    w = np.array(wins)
    assert (got['status'] == 0).all()
    assert np.abs(got['lo'] - w[:, 0]).max() < 60 and np.abs(got['hi'] - w[:, 1]).max() < 60


# accuracy on synthetic truth (noise 0.15); DESIGN.md section 4.5 records the measured figures
def test_accuracy_on_synthetic_truth(built_lib):
    locus = synth.make_locus('HD', seed=10)
    eng, stas, ids = _engine(locus)
    sigs, wins, rev, truth = _whole_reads(locus, 2000, seed=14, pad=(4_000, 20_000))
    aut = [ids[int(r)] for r in rev]
    got = _locate(eng, sigs, aut)
    w = np.array(wins)
    d_lo, d_hi = got['lo'] - w[:, 0], got['hi'] - w[:, 1]
    err = np.maximum(np.abs(d_lo), np.abs(d_hi))
    print('locate accuracy: found', int((got['status'] == 0).sum()), 'of', len(sigs),
          '| end error p50/p99/max', np.percentile(err, 50), np.percentile(err, 99), err.max())
    assert (got['status'] == 0).all()
    assert np.percentile(err, 99) <= 40 and err.max() <= 120
    # the calls on the located windows against the calls on the true windows
    on_true = eng.call_batch([s[a:b + 1] for s, (a, b) in zip(sigs, wins)], aut, rev)
    on_loc = eng.call_batch([s[a:b + 1] for s, a, b in zip(sigs, got['lo'], got['hi'])], aut, rev)
    same = np.mean([len(x.resc_seq) == len(y.resc_seq) for x, y in zip(on_true, on_loc)])
    print('locate accuracy: same allele length as on the true window', same)
    assert same >= 0.95


def _fixture():
    z = np.load(os.path.join(GOLD, 'c1_bundled.npz'))
    raws = [np.cumsum(z[f'raw_delta{i}'].astype(np.int64)).astype(np.int16) for i in range(len(z['names']))]
    return z, raws


def _bundled_wrapper(z):
    from warpstr_b200.wrapper import CallerWrapper, Locus, flanks_from_template
    locus = Locus(name='Human_STR_1108232', sequence=str(z['sequence']), flank_length=int(z['flank_length']))
    return CallerWrapper(locus, threads=2, flanks=flanks_from_template(str(z['left']), str(z['right'])))


def test_bundled_whole_reads_normalise_like_numpy(built_lib):
    from oracle import normalize_oracle as no
    from warpstr_b200.normalize import normalize_windows
    z, raws = _fixture()
    got = normalize_windows(raws, [(0, len(r) - 1) for r in raws], 'Brute')
    for i, raw in enumerate(raws):
        assert np.array_equal(got[i], no.get_data_processed(raw, (0, len(raw) - 1))), i


def test_bundled_reads_located_and_called(built_lib):
    from oracle import normalize_oracle as no
    z, raws = _fixture()
    cw = _bundled_wrapper(z)
    rev = [bool(r) for r in z['reverse']]
    loc = cw.locate_raw(raws, rev)
    assert (loc['status'] == 0).all()
    assert np.abs(loc['lo'] - z['l_start_raw']).max() <= 50 and np.abs(loc['hi'] - z['r_end_raw']).max() <= 50
    # the kernel against the oracle on the same whole reads
    sigs = [no.get_data_processed(raw, (0, len(raw) - 1)) for raw in raws]
    _same_as_oracle(loc, sigs, [cw.rev_sta if r else cw.temp_sta for r in rev], 4)
    res = cw.run_raw(raws, None, rev)
    assert [len(r.seq) for r in res] == z['len1'].tolist()
    assert [len(r.resc_seq) for r in res] == z['len2'].tolist()
    assert sorted(set(len(r.resc_seq) for r in res)) == [40, 44]
    assert np.array_equal(cw.engine.last_located['lo'], loc['lo'])


def test_bundled_reads_main_wrapper_without_windows(built_lib, tmp_path):
    """fast5 files + a caller-only CSV without window columns -> overview with results and located windows."""
    import pandas as pd
    from warpstr_b200 import caller_only
    from warpstr_b200.wrapper import Locus, flanks_from_template, main_wrapper
    z, raws = _fixture()
    names = [str(n) for n in z['names']]
    paths = []
    for k in range(2):
        p = str(tmp_path / f'run{k}.fast5')
        hw.write_multi(p, {n: raws[i] for i, n in enumerate(names) if i % 2 == k}, 'vbz0', chunk=4000)
        paths.append(p)
    csv_path = str(tmp_path / 'reads.csv')
    with open(csv_path, 'w') as fh:
        fh.write('fast5_path,locus,read_name,reverse\n')
        for i, n in enumerate(names):
            fh.write(f'{paths[i % 2]},LOC,{n},{bool(z["reverse"][i])}\n')
    out = str(tmp_path / 'out')
    caller_only.prepare(out, csv_path)
    locus = Locus(name='LOC', sequence=str(z['sequence']), flank_length=int(z['flank_length']),
                  path=os.path.join(out, 'LOC'))
    main_wrapper(locus, flanks=flanks_from_template(str(z['left']), str(z['right'])))
    df = pd.read_csv(os.path.join(out, 'LOC', 'overview.csv')).set_index('read_name').loc[names]
    assert df['results'].tolist() == z['len2'].tolist() and df['orig'].tolist() == z['len1'].tolist()
    assert np.abs(df['l_start_raw'].to_numpy() - z['l_start_raw']).max() <= 50
    assert np.abs(df['r_end_raw'].to_numpy() - z['r_end_raw']).max() <= 50


def test_main_wrapper_not_found_row_has_no_result(built_lib, tmp_path):
    """One row with a window, one to locate, one that holds only filler: one warning names the lost read, its
    result cells stay empty, the others are called."""
    import pandas as pd
    from warpstr_b200 import caller_only
    from warpstr_b200.wrapper import Locus, flanks_from_template, main_wrapper
    locus = synth.make_locus('HD', seed=41)
    reads = synth.make_reads(locus, 2, seed=42, noise=0.15)
    rng = np.random.default_rng(43)
    raws, wins = {}, {}
    for i, r in enumerate(reads):
        raw, lo, hi = synth.to_raw_int16(rng, r.signal, pad=20_000, spike_rate=1e-4)
        raws[f'r{i}'] = raw
        wins[f'r{i}'] = (lo, hi)
    filler, _, _ = synth.to_raw_int16(rng, _filler(rng, 20_000, synth.get_pore_model()), pad=2000)
    raws['lost'] = filler
    p = str(tmp_path / 'run.fast5')
    hw.write_multi(p, raws, 'vbz0', chunk=4000)
    csv_path = str(tmp_path / 'reads.csv')
    rev = {'r0': reads[0].reverse, 'r1': reads[1].reverse, 'lost': False}
    with open(csv_path, 'w') as fh:
        fh.write('fast5_path,locus,read_name,reverse,l_start_raw,r_end_raw\n')
        fh.write(f'{p},LOC,r0,{rev["r0"]},{wins["r0"][0]},{wins["r0"][1]}\n')
        fh.write(f'{p},LOC,r1,{rev["r1"]},,\n')
        fh.write(f'{p},LOC,lost,False,,\n')
    out = str(tmp_path / 'out')
    caller_only.prepare(out, csv_path)
    loc = Locus(name='LOC', sequence=locus.sequence, flank_length=locus.flank_length, path=os.path.join(out, 'LOC'))
    with pytest.warns(RuntimeWarning, match='lost'):
        main_wrapper(loc, flanks=flanks_from_template(locus.left, locus.right))
    df = pd.read_csv(os.path.join(out, 'LOC', 'overview.csv')).set_index('read_name')
    assert df.loc['r0', 'results'] > 0 and df.loc['r1', 'results'] > 0
    assert pd.isna(df.loc['lost', 'results']) and pd.isna(df.loc['lost', 'l_start_raw'])
    assert abs(df.loc['r1', 'l_start_raw'] - wins['r1'][0]) < 60 and abs(df.loc['r1', 'r_end_raw'] - wins['r1'][1]) < 60
    assert (df.loc['r0', 'l_start_raw'], df.loc['r0', 'r_end_raw']) == wins['r0']
