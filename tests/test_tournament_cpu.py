"""CPU: the ctypes mirror of bz_tournament_state has the C compiler's layout, and the tournament's rating fit."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "betazero_b200.h")


def test_tournament_state_layout_matches_the_c_compiler(tmp_path):
    from betazero_b200._lib import BzMatchState, BzTournamentState

    fields = [n for n, _ in BzTournamentState._fields_]
    inner = [n for n, _ in BzMatchState._fields_]
    prog = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', "int main(void){",
            'printf("%zu\\n", sizeof(bz_tournament_state));']
    prog += [f'printf("%zu\\n", offsetof(bz_tournament_state, {f}));' for f in fields]
    prog += [f'printf("%zu\\n", offsetof(bz_tournament_state, match.{f}));' for f in inner]
    prog += ['printf("%d\\n", BZ_MAX_ENTRANTS);', "return 0;}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(prog))
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-o", str(exe), str(src)])
    vals = [int(v) for v in subprocess.check_output([str(exe)], text=True).split()]
    exp = [C.sizeof(BzTournamentState)] + [getattr(BzTournamentState, f).offset for f in fields]
    exp += [getattr(BzMatchState, f).offset for f in inner]
    from betazero_b200 import tournament

    assert vals == exp + [tournament.MAX_ENTRANTS]


def test_nested_match_state_writes_through():
    """Tournament fills the match part through ``state.match``: a view into the same buffer, not a copy"""
    from betazero_b200._lib import BzTournamentState

    s = BzTournamentState()
    m = s.match
    m.n_games, m.counters = 42, 1234
    assert s.match.n_games == 42 and s.match.counters == 1234 and C.addressof(m) == C.addressof(s)


def test_two_entrants_equal_the_closed_form_with_the_virtual_draw():
    from betazero_b200.match import elo
    from betazero_b200.tournament import fit_ratings

    for scores in ([1.0, 0.75, 0.5, 0.5, 0.25], [1.0] * 7, [0.0, 0.25], [0.5] * 3):
        n, s = len(scores), float(np.mean(scores))
        r, se = fit_ratings(2, [(0, 1)], [scores])
        assert r[0] == 0.0 and se[0] == 0.0
        assert r[1] == pytest.approx(-elo((n * s + 0.5) / (n + 1)), abs=1e-9)  # entrant 0's score s: r1 - r0 = -elo
        p = (n * s + 0.5) / (n + 1)  # binomial information of n + 1 pairs at the fitted score
        assert se[1] == pytest.approx(1.0 / math.sqrt((n + 1) * p * (1 - p)) / (math.log(10) / 400), rel=1e-9)


def test_swapping_entrants_negates_the_ratings():
    from betazero_b200.tournament import fit_ratings

    r, _ = fit_ratings(2, [(0, 1)], [[0.75, 1.0, 0.5]])
    r2, _ = fit_ratings(2, [(1, 0)], [[0.75, 1.0, 0.5]])
    assert r2[1] == pytest.approx(-r[1], abs=1e-9) and r[1] < 0
    rng = np.random.default_rng(0)
    pairs = [(0, 1), (1, 2), (0, 2), (2, 3)]
    sc = [rng.choice([0, 0.25, 0.5, 0.75, 1.0], 20) for _ in pairs]
    a, _ = fit_ratings(4, pairs, sc)
    b, _ = fit_ratings(4, [(j, i) for i, j in pairs], [1.0 - x for x in sc])  # the same games, seen from the other side
    assert np.allclose(a, b, atol=1e-9)
    c, _ = fit_ratings(4, pairs, [1.0 - x for x in sc])  # every result reversed
    assert np.allclose(c, -a, atol=1e-9)


def test_all_draws_give_zeros_and_a_clean_sweep_stays_finite():
    from betazero_b200.tournament import fit_ratings

    pairs = [(i, j) for i in range(4) for j in range(i + 1, 4)]
    r, se = fit_ratings(4, pairs, [[0.5] * 10 for _ in pairs])
    assert np.allclose(r, 0.0, atol=1e-12) and (se[1:] > 0).all()
    r, se = fit_ratings(4, pairs, [[1.0] * 50 for _ in pairs])  # lower id always wins
    assert np.isfinite(r).all() and np.isfinite(se).all()
    assert r[0] > r[1] > r[2] > r[3]


def test_exact_expected_scores_recover_known_ratings():
    from betazero_b200.tournament import fit_ratings

    true = np.array([0.0, 100.0, -50.0, 200.0, 35.0])
    pairs = [(i, j) for i in range(5) for j in range(i + 1, 5)]
    n = 200000
    sc = [np.full(n, 1.0 / (1.0 + 10 ** ((true[j] - true[i]) / 400))) for i, j in pairs]
    r, se = fit_ratings(5, pairs, sc)
    # the virtual draws pull differences towards 0 by O(1/n) of them
    assert np.allclose(r, true, atol=0.05) and np.abs(r).max() < np.abs(true).max()
    assert (se[1:] < 2.0).all()


def test_a_disconnected_pairing_graph_raises():
    from betazero_b200.tournament import fit_ratings

    with pytest.raises(ValueError, match="connect"):
        fit_ratings(4, [(0, 1), (2, 3)], [[0.5], [0.5]])
    with pytest.raises(ValueError, match="connect"):
        fit_ratings(3, [(0, 1), (1, 2)], [[0.5], []])  # a pairing without a finished pair does not connect


def test_tournament_refuses_bad_arguments_before_touching_a_device():
    from betazero_b200.tournament import Tournament

    two = [(None, 16), (None, 16)]
    with pytest.raises(ValueError, match="entrants"):
        Tournament([(None, 16)], 2)
    with pytest.raises(ValueError, match="entrants"):
        Tournament([(None, 16)] * 65, 2)
    with pytest.raises(ValueError, match="multiple"):
        Tournament([(None, 16), (None, 18)], 2, n_leaves=4)
    with pytest.raises(ValueError, match="even"):
        Tournament(two, 3)
    with pytest.raises(ValueError, match="twice"):
        Tournament(two, 2, pairings=[(0, 1), (1, 0)])
    with pytest.raises(ValueError, match="different"):
        Tournament(two, 2, pairings=[(0, 0)])
    with pytest.raises(ValueError, match="connect"):
        Tournament([(None, 16)] * 4, 2, pairings=[(0, 1), (2, 3)])
    with pytest.raises(ValueError, match="65536"):
        Tournament(two, 65536)


def test_loop_checkpoint_path_keeps_one_file_per_iteration():
    from betazero_b200.loop import checkpoint_path

    assert checkpoint_path("ck/it{iteration}.pt", 3) == "ck/it3.pt"
    assert checkpoint_path("ck/net.pt", 3) == "ck/net.pt"
