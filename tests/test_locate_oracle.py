"""CPU: the STR window search of oracle/locate_oracle.c (wso_locate) against an enumeration of every path
on tiny automata and signals.  Values are multiples of 1/8, so every sum is exact and ties are real ties:
the expected window is the one the recurrence's order picks among the optimal paths (stay, then the
incoming states in list order, then a start; the earliest end row)."""
import itertools
from types import SimpleNamespace

import numpy as np
import pytest

from oracle import locate as lo_oracle


def _aut(values, incoming, endstate):
    ip = np.zeros(len(values) + 1, dtype=np.int32)
    ip[1:] = np.cumsum([len(x) for x in incoming])
    ii = np.array([p for x in incoming for p in x], dtype=np.int32)
    return SimpleNamespace(values=np.asarray(values, dtype=np.float64), seq_idx=np.arange(len(values), dtype=np.int32),
                           in_ptr=ip, in_idx=ii, endstate=int(endstate))


def _brute(x, a, m, lam):
    """(lo, hi, score, status) from every path, the recurrence's tie order made explicit: a path is its
    backward choice sequence (0 stay, 1 + k the k-th incoming state, a large code for the start), and of
    the optimal paths ending on the earliest optimal row the lexicographically smallest one wins."""
    inc = [list(a.in_idx[a.in_ptr[j]:a.in_ptr[j + 1]]) for j in range(len(a.values))]
    c = lambda t, j: abs(x[t] - a.values[j]) - lam
    START = 1 << 30

    def paths(i, j):            # (cost, choices, start row) of every path that ends in cell (i, j)
        out = []
        if j == 0:
            out.append((c(i, 0), (START,), i))
        if i >= 1:
            for cost, ch, s in paths(i - 1, j):
                out.append((cost + c(i, j), (0,) + ch, s))
        if i >= m:
            for k, p in enumerate(inc[j]):
                for cost, ch, s in paths(i - m, p):
                    out.append((cost + sum(c(t, p) for t in range(i - m + 1, i)) + c(i, j), (1 + k,) + ch, s))
        return out

    best = None
    for i in range(len(x)):
        ps = paths(i, a.endstate)
        if not ps:
            continue
        e = min(p[0] for p in ps)
        if best is None or e < best[2]:
            win = min((p for p in ps if p[0] == e), key=lambda p: p[1])
            best = (win[2], i, e)
    if best is None:
        return -1, -1, np.inf, 2
    return best[0], best[1], best[2], 0 if best[2] < 0 else 1


def _check(x, a, m, lam):
    want = _brute(np.asarray(x, dtype=np.float64), a, m, lam)
    got = lo_oracle.locate(np.asarray(x, dtype=np.float64), a, m, lam)
    assert got == want, (got, want)
    return got


CHAIN3 = _aut([0.0, 1.0, 2.0], [[], [0], [1]], 2)


def test_free_start_and_end():
    # the flank-repeat-flank chain sits in the middle of filler that matches nothing
    x = [5, 5, 5, 0, 0, 1, 1, 2, 2, 5, 5]
    lo, hi, score, st = _check(x, CHAIN3, 2, 0.25)
    assert (lo, hi, st) == (3, 8, 0) and score == -6 * 0.25


def test_dwell_is_enforced():
    # one sample of state 1 is too short for m = 2: the path has to spend two rows there
    x = [0, 0, 1, 2, 2]
    lo, hi, _, st = _check(x, CHAIN3, 2, 0.25)
    assert st == 0 and (lo, hi) == (0, 4)
    _check(x, CHAIN3, 3, 0.25)


def test_tie_order_of_incoming_states():
    # state 2 is reached from 0 or from 1 at the same cost: the first incoming state in list order wins
    a = _aut([0.0, 0.0, 1.0], [[], [0], [1, 0]], 2)
    _check([0, 0, 0, 0, 1, 1], a, 2, 0.5)
    b = _aut([0.0, 0.0, 1.0], [[], [0], [0, 1]], 2)
    _check([0, 0, 0, 0, 1, 1], b, 2, 0.5)


def test_start_versus_stay_tie():
    # x[1] is exactly lam from state 0's level: staying and starting anew at row 1 both cost c_1(0) + (0 or
    # L[0][0] = 0); stay is tried first, so the window starts at row 0
    a = _aut([0.0, 2.0], [[], [0]], 1)
    lo, hi, score, st = _check([0.25, 0.5, 0.5, 2, 2, 2, 2], a, 2, 0.25)
    assert st == 0 and lo == 0


def test_not_found_and_no_path():
    # every sample far from every level: the best window costs more than nothing
    _, _, score, st = _check([9, 9, 9, 9, 9, 9], CHAIN3, 2, 0.25)
    assert st == 1 and score > 0
    # shorter than the automaton's shortest path (2 + 2 + 1 rows): no path at all
    assert _check([0, 1, 2], CHAIN3, 2, 0.25)[3] == 2


@pytest.mark.parametrize('seed', range(40))
def test_random_automata_against_enumeration(seed):
    rng = np.random.default_rng([seed, 0x10CA7E])
    S = int(rng.integers(2, 5))
    incoming = [[]] + [rng.permutation(rng.choice(j, size=int(rng.integers(1, min(j, 2) + 1)), replace=False)).tolist()
                       for j in range(1, S)]
    if rng.random() < 0.3 and S > 2:          # a back edge (loops such as (CAG) make these)
        incoming[1].append(S - 1)
    values = rng.integers(0, 4, size=S) / 4.0
    a = _aut(values, incoming, S - 1)
    m = int(rng.integers(2, 4))
    x = rng.integers(0, 6, size=int(rng.integers(S, 11))) / 4.0 - 0.25
    _check(x, a, m, float(rng.integers(0, 4)) / 8.0)


def test_every_short_signal():
    # every signal of six samples over the chain's three levels
    for x in itertools.product([0.0, 1.0, 2.0], repeat=6):
        lo, hi, score, st = _check(list(x), CHAIN3, 2, 0.5)
        if st != 2:
            assert 0 <= lo <= hi < 6
