"""GPU: a panel's reads found in whole reads by their flanks (DESIGN.md section 4.6).  locate_group_kernel's
searches equal wstr_locate_batch's bit for bit (and so the C oracle's), the device hit list is assign.choose_loci
of them, reads of synthetic loci are assigned to their locus and strand and nothing else is, and files with no
read names give the bundled reads' overview and calls."""
import os
import uuid

import numpy as np
import pytest

import _h5write as hw
import _pod5write as pw
from warpstr_b200 import synth

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), 'golden')


def _filler(rng, n, pm):
    """~n samples of squiggled random sequence."""
    return synth.squiggle(rng, synth.random_flank(rng, n // 9 + 8), pm)[:n]


def _embed(rng, sig, pad, pm):
    a, b = (int(x) for x in rng.integers(pad[0], pad[1] + 1, size=2))
    return np.concatenate((_filler(rng, a, pm), sig, _filler(rng, b, pm)))


def _flanks(locus):
    from warpstr_b200.wrapper import flanks_from_template
    return flanks_from_template(locus.left, locus.right)


def _bits(x):
    return np.asarray(x, dtype=np.float64).view(np.int64)


def _device(sigs, eng):
    from warpstr_b200.caller import pack_signals
    host, off, lengths = pack_signals(sigs)
    return host.to(eng.device), off, lengths


def _parity(mv, units, sigs):
    """wstr_assign_batch with d_table against wstr_locate_batch on every (read, automaton); the hit list against
    choose_loci of the table."""
    import torch
    from warpstr_b200 import _lib
    from warpstr_b200.assign import choose_loci
    from warpstr_b200.caller import CallerEngine, hit_arrays
    from warpstr_b200.config import CallerConfig
    eng = CallerEngine(CallerConfig(min_values_per_state=mv))
    ids = [eng.add_automaton(a, 110) for u in units for a in u]
    auts = [eng.automata[i] for i in ids]
    d_sig, off, lengths = _device(sigs, eng)
    n, A = len(sigs), len(auts)
    d_table = torch.zeros(20 * n * A, dtype=torch.uint8, device=eng.device)
    d_hits = torch.zeros(max(n * A // 4, 1) * _lib.ASSIGN_HIT.itemsize, dtype=torch.uint8, device=eng.device)
    d_n = torch.zeros(1, dtype=torch.int32, device=eng.device)
    ws = torch.empty(_lib.assign_workspace_bytes(auts, n), dtype=torch.uint8, device=eng.device)
    _lib.assign_batch(auts, d_sig, off, lengths, 0.35, d_table, d_hits, d_n, ws)
    lo, hi, score, status = _lib.split_table(d_table.cpu().numpy(), n, A)
    # the same entries through wstr_locate_batch, one (read, automaton) per entry
    ra = np.tile(np.arange(A, dtype=np.int32), n)
    rd = np.repeat(np.arange(n), A)
    m = n * A
    d_i = torch.empty((3, m), dtype=torch.int32, device=eng.device)
    d_sc = torch.empty(m, dtype=torch.float64, device=eng.device)
    lws = torch.empty(_lib.locate_workspace_bytes(auts, m), dtype=torch.uint8, device=eng.device)
    _lib.locate_batch(auts, ra, d_sig, off[rd], lengths[rd], 0.35, d_i[0], d_i[1], d_sc, d_i[2], lws)
    want = d_i.cpu().numpy().reshape(3, n, A)
    assert np.array_equal(status, want[2]) and np.array_equal(lo, want[0]) and np.array_equal(hi, want[1])
    assert np.array_equal(_bits(score), _bits(d_sc.cpu().numpy().reshape(n, A)))
    k = int(d_n.cpu()[0])
    got = hit_arrays(d_hits[:k * _lib.ASSIGN_HIT.itemsize].cpu().numpy().view(_lib.ASSIGN_HIT))
    ref = choose_loci(lo, hi, score, status)
    for f in ref:
        assert np.array_equal(got[f].view(np.int64) if got[f].dtype == np.float64 else got[f],
                              ref[f].view(np.int64) if ref[f].dtype == np.float64 else ref[f]), f
    return status, ref


def _units(locus, pm):
    """Two loci's worth of automata for one synthetic locus: its two full automata and its four flank chains."""
    from warpstr_b200.assign import flank_chains
    from warpstr_b200.automata import StateAutomata
    full = [StateAutomata(locus.template_regex, pm), StateAutomata(locus.reverse_regex, pm)]
    tl, tr, rl, rr = flank_chains(_flanks(locus), pm)
    return [[full[0], full[1], tl, tr], [rl, rr, full[0], full[1]], [tl, tr, rl, rr]]


@pytest.mark.parametrize('mv', [2, 4, 8])
def test_group_kernel_matches_locate_batch(built_lib, mv):
    """Five loci (HD, FMR1, DM2, (CAN), C9orf72) in one launch: several groups per read, every group several
    automata; on-target reads of two strands, a pure filler read, reads shorter than any path."""
    pm = synth.get_pore_model()
    names = ['HD', 'FMR1', 'DM2', 'CAN', 'C9ORF72_100']
    loci = [synth.make_locus(nm, seed=80 + k) for k, nm in enumerate(names)]
    units = [u for L in loci for u in _units(L, pm)]
    rng = np.random.default_rng(81)
    sigs = []
    for k, L in enumerate(loci):
        sigs += [_embed(rng, r.signal, (500, 4000), pm) for r in synth.make_reads(L, 2, seed=90 + k)]
    sigs += [_filler(rng, 12_000, pm), sigs[0][:40], sigs[1][:3]]
    status, hits = _parity(mv, units, sigs)
    assert (status[-2:] == 2).all() and not (status[-3] == 0).any()
    if mv == 4:          # every on-target read is found on its own chains unit
        assert set(zip(hits['read'].tolist(), hits['locus'].tolist())) >= {(r, 3 * (r // 2) + 2) for r in range(10)}


@pytest.mark.parametrize('mv', [4, 8])
def test_group_kernel_workspace_rings(built_lib, mv):
    """A locus whose automata do not fit the group budget: its rings live in the workspace, next to groups that
    keep them in shared memory."""
    from warpstr_b200.automata import StateAutomata
    pm = synth.get_pore_model()
    rng = np.random.default_rng(82)
    L = synth.make_locus('HD', seed=83)
    long_seq = synth.random_flank(rng, 1500)
    big = [StateAutomata(long_seq, pm), StateAutomata(synth.random_flank(rng, 1200), pm)]
    units = _units(L, pm)[2:] + [[big[0], big[1]] + _units(L, pm)[2][:2]] + _units(L, pm)[:1]
    sigs = [_embed(rng, r.signal, (500, 3000), pm) for r in synth.make_reads(L, 3, seed=84)]
    sigs.append(_embed(rng, synth.squiggle(rng, long_seq, pm), (1000, 2000), pm))
    status, _ = _parity(mv, units, sigs)
    assert status[3, 4] == 0          # the long chain found in the read that carries it


def _panel(loci, mv=4):
    from warpstr_b200.assign import Panel
    return Panel([(L.name, _flanks(L)) for L in loci], min_values_per_state=mv)


def _engine(mv=4):
    from warpstr_b200.caller import CallerEngine
    from warpstr_b200.config import CallerConfig
    return CallerEngine(CallerConfig(min_values_per_state=mv))


def _accuracy(noise, n_on, n_off):
    pm = synth.get_pore_model()
    names = ['HD', 'FMR1', 'DM2', 'CAN']
    loci = [synth.make_locus(nm, seed=300 + k) for k, nm in enumerate(names)]
    rng = np.random.default_rng([int(noise * 100), 301])
    sigs, truth_locus, truth_rev = [], [], []
    for k, L in enumerate(loci):
        for r in synth.make_reads(L, n_on, seed=310 + k, noise=noise):
            sigs.append(_embed(rng, r.signal, (2000, 10_000), pm))
            truth_locus.append(k)
            truth_rev.append(int(r.reverse))
    for _ in range(n_off):
        sigs.append(_filler(rng, int(rng.integers(4000, 24_000)), pm))
        truth_locus.append(-1)
        truth_rev.append(-1)
    eng = _engine()
    d_sig, off, lengths = _device(sigs, eng)
    hits = eng.assign_packed(d_sig, off, lengths, _panel(loci))
    truth_locus, truth_rev = np.array(truth_locus), np.array(truth_rev)
    on = truth_locus >= 0
    right = (truth_locus[hits['read']] == hits['locus']) & (truth_rev[hits['read']] == hits['strand'])
    wrong_locus = int(((truth_locus[hits['read']] != hits['locus']) & on[hits['read']]).sum())
    off_hits = int((~on[hits['read']]).sum())
    n_right = len(set(hits['read'][right].tolist()))
    print(f'assignment, noise {noise}: {n_right} of {int(on.sum())} on-target reads on their locus and strand, '
          f'{wrong_locus} hits on a wrong locus, {off_hits} hits of {n_off} off-target reads, '
          f'{int((truth_locus[hits["read"]] == hits["locus"]).sum()) - int(right.sum())} on the wrong strand')
    return n_right, int(on.sum()), wrong_locus, off_hits, len(hits['read']), int(right.sum())


def test_assignment_on_synthetic_truth(built_lib):
    n_right, n_on, wrong_locus, off_hits, n_hits, n_right_hits = _accuracy(0.15, 500, 2000)
    assert n_right == n_on and wrong_locus == 0 and off_hits == 0 and n_hits == n_right_hits == n_on
    _accuracy(0.30, 500, 2000)


def test_same_motif_other_locus(built_lib):
    """Two loci of the same motif, different flanks; reads with a 1 000-unit expansion of either: each read is
    assigned to its own locus only (the expansion matches the other locus's repeat automaton, never its flanks)."""
    pm = synth.get_pore_model()
    loci = [synth.make_locus('CAN', seed=400 + k) for k in range(2)]
    loci[1].name = 'CAN_b'
    rng = np.random.default_rng(401)
    from warpstr_b200.templates import reverse_complement
    sigs, truth = [], []
    for k, L in enumerate(loci):
        for j in range(12):
            seq = L.left + 'CAG' * 1000 + L.right
            rev = j % 2 == 1
            sigs.append(_embed(rng, synth.squiggle(rng, reverse_complement(seq) if rev else seq, pm), (2000, 6000), pm))
            truth.append((k, int(rev)))
    eng = _engine()
    d_sig, off, lengths = _device(sigs, eng)
    hits = eng.assign_packed(d_sig, off, lengths, _panel(loci))
    got = list(zip(hits['read'].tolist(), hits['locus'].tolist(), hits['strand'].tolist()))
    assert got == [(r, k, s) for r, (k, s) in enumerate(truth)]


def _fixture():
    z = np.load(os.path.join(GOLD, 'c1_bundled.npz'))
    raws = [np.cumsum(z[f'raw_delta{i}'].astype(np.int64)).astype(np.int16) for i in range(len(z['names']))]
    return z, raws


def test_files_to_overview_to_calls(built_lib, tmp_path):
    """The bundled ten reads among 200 off-target reads, in one POD5 and one multi-read fast5, no read names: exactly
    the ten are assigned, with their strands; main_wrapper on the overview gives the calls of the same reads listed
    by name without strands (test_gpu_strand); both files give the same overview."""
    import warnings
    import pandas as pd
    from test_gpu_strand import OUT_FILES, _bundled_locus, _main_wrapper
    from warpstr_b200.assign import assign_files
    from warpstr_b200.config import Config, LocusConfig
    from warpstr_b200.wrapper import Locus, flanks_from_template, main_wrapper
    z, raws = _fixture()
    names = [str(n) for n in z['names']]
    pm = synth.get_pore_model()
    rng = np.random.default_rng(500)
    reads = {}
    off = {str(uuid.UUID(bytes=rng.bytes(16), version=4)): synth.to_raw_int16(rng, _filler(rng, 20_000, pm), pad=2000)[0]
           for _ in range(200)}
    order = list(off) + names
    rng.shuffle(order)
    for n in order:
        reads[n] = raws[names.index(n)] if n in names else off[n]
    p5, f5 = str(tmp_path / 'run.pod5'), str(tmp_path / 'run.fast5')
    pw.write(p5, reads, rows=lambda i, n: 1 + i % 2, seed=1)
    hw.write_multi(f5, reads, 'vbz0', chunk=4000)
    locus = _bundled_locus(z)
    name = 'Human_STR_1108232'
    flanks = {name: flanks_from_template(locus.left, locus.right)}
    overviews = {}
    for tag, path in (('pod5', p5), ('fast5', f5)):
        cfg = Config(output=str(tmp_path / f'out_{tag}'), loci=[LocusConfig(name=name, sequence=locus.sequence)])
        counts = assign_files(cfg, [path], flanks=flanks, chunk_reads=64)
        assert counts == {name: 10}
        ov = os.path.join(cfg.output, name, 'overview.csv')
        with open(ov) as fh:
            overviews[tag] = fh.read().replace(path, 'RUN')
        df = pd.read_csv(ov)
        assert sorted(df['read_name']) == sorted(names)
        truth = dict(zip(names, (bool(r) for r in z['reverse'])))
        assert [truth[n] for n in df['read_name']] == df['reverse'].tolist()
        assert df['l_start_raw'].isna().all() and df['r_end_raw'].isna().all()
    assert overviews['pod5'] == overviews['fast5']
    # main_wrapper on the assigned overview = the named route with empty strands and windows
    path = os.path.join(str(tmp_path / 'out_fast5'), name)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        main_wrapper(Locus(name=name, sequence=locus.sequence, flank_length=locus.flank_length, path=path),
                     flanks=flanks[name])
    df = pd.read_csv(os.path.join(path, 'overview.csv')).set_index('read_name').loc[names]
    assert df['results'].tolist() == z['len2'].tolist() and df['orig'].tolist() == z['len1'].tolist()
    assert sorted(set(df['results'])) == [40, 44]
    named, files = _main_wrapper(tmp_path, 'named', locus, [(f5, n, '', '', '') for n in names])
    named = named.loc[names]
    for c in ('reverse', 'l_start_raw', 'r_end_raw', 'results', 'orig', 'dtw_cost1', 'dtw_cost2'):
        assert df[c].tolist() == named[c].tolist(), c
    for f in ('predictions/sequences/all.fasta',):
        with open(os.path.join(path, f), 'rb') as fh:
            mine = fh.read()
        assert sorted(mine.split(b'>')) == sorted(files[f].split(b'>')), f
