"""Flank-chain score distributions on the C oracle (oracle/locate_oracle.c), no GPU: the numbers of DESIGN.md
section 4.6.  Four synthetic loci (HD, FMR1, DM2, (CAN)), their four flank chains each; 200 off-target reads of
random sequence (20 000-60 000 samples) and 50 reads per locus between 2 000-10 000 filler samples either side
(noise 0.15, min_values_per_state 4, offset 0.35).  Prints the score distributions and how many reads pass the
rule of assign.choose_loci for which locus.

    python scripts/calibrate_assign.py
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    from oracle import locate as lo_oracle
    from warpstr_b200 import synth
    from warpstr_b200.assign import Panel, choose_loci
    from warpstr_b200.wrapper import flanks_from_template
    pm = synth.get_pore_model()
    loci = [synth.make_locus(n, seed=100 + k) for k, n in enumerate(('HD', 'FMR1', 'DM2', 'CAN'))]
    panel = Panel([(L.name, flanks_from_template(L.left, L.right)) for L in loci])
    rng = np.random.default_rng(7)

    def filler(n):
        return synth.squiggle(rng, synth.random_flank(rng, n // 9 + 8), pm)[:n]

    sigs = [filler(int(rng.integers(20_000, 60_001))) for _ in range(200)]
    truth = [(-1, -1)] * 200
    for k, L in enumerate(loci):
        for r in synth.make_reads(L, 50, seed=200 + k):
            a, b = (int(x) for x in rng.integers(2000, 10_001, size=2))
            sigs.append(np.concatenate((filler(a), r.signal, filler(b))))
            truth.append((k, int(r.reverse)))
    A, n = len(panel.chains), len(sigs)
    lo, hi, score, status = (x.reshape(n, A) for x in lo_oracle.locate_batch(
        [s for s in sigs for _ in range(A)], panel.chains * n, 4, threads=os.cpu_count() or 8))
    truth = np.array(truth)
    off = truth[:, 0] < 0
    own = np.zeros((n, A), dtype=bool)
    for r in np.flatnonzero(~off):
        own[r, 4 * truth[r, 0] + 2 * truth[r, 1] + np.arange(2)] = True
    other_strand = np.zeros((n, A), dtype=bool)
    for r in np.flatnonzero(~off):
        other_strand[r, 4 * truth[r, 0] + 2 * (1 - truth[r, 1]) + np.arange(2)] = True
    q = lambda x: ' '.join(f'{v:.1f}' for v in np.percentile(x, [0, 1, 50, 99, 100]))   # noqa: E731
    print('flank scores, min p1 p50 p99 max')
    print('  off-target reads, every chain:          ', q(score[off]), f'found {int((status[off] == 0).sum())}')
    print('  on-target reads, own locus and strand:  ', q(score[own]))
    print('  on-target reads, own locus, other strand:', q(score[other_strand]))
    print('  on-target reads, other loci:            ', q(score[~off[:, None] & ~own & ~other_strand]))
    hits = choose_loci(lo, hi, score, status)
    rd, lc, st = hits['read'], hits['locus'], hits['strand']
    print(f'hits: {int((~off[rd]).sum())} on-target ({int(((truth[rd, 0] == lc) & (truth[rd, 1] == st)).sum())} on '
          f'their locus and strand, of {int((~off).sum())}), {int(off[rd].sum())} off-target')


if __name__ == '__main__':
    main()
