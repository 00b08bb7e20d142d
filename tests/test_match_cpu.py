"""CPU: the ctypes mirror of bz_match_state has the C compiler's layout, and the match score's Elo arithmetic."""
import ctypes as C
import math
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "betazero_b200.h")


def test_match_state_layout_matches_the_c_compiler(tmp_path):
    from betazero_b200._lib import BzMatchState

    fields = [n for n, _ in BzMatchState._fields_]
    prog = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', "int main(void){",
            'printf("%zu\\n", sizeof(bz_match_state));']
    prog += [f'printf("%zu\\n", offsetof(bz_match_state, {f}));' for f in fields]
    prog += ['printf("%d %d %d\\n", BZ_MATCH_RUNNING, BZ_MATCH_MAX_PLIES, BZ_MATCH_TREES_PER_PAIR);', "return 0;}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(prog))
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-o", str(exe), str(src)])
    vals = [int(v) for v in subprocess.check_output([str(exe)], text=True).split()]
    assert vals[:-3] == [C.sizeof(BzMatchState)] + [getattr(BzMatchState, f).offset for f in fields]
    from betazero_b200 import match

    assert vals[-3:] == [match.RUNNING, match.MAX_PLIES, match.TREES_PER_PAIR]


def test_elo_of_a_score():
    from betazero_b200.match import elo

    assert elo(0.5) == 0.0
    assert elo(0.75) == pytest.approx(400 * math.log10(3))  # 190.85: 3 to 1 odds
    assert elo(0.25) == pytest.approx(-400 * math.log10(3))
    assert elo(1.0) == math.inf and elo(0.0) == -math.inf


def test_elo_interval_from_pair_scores():
    from betazero_b200.match import elo_summary

    # four pairs: mean 1/2; sample variance (1/4 + 0 + 0 + 1/4) / 3 = 1/6; standard error sqrt(1/6 / 4) = sqrt(1/24)
    r = elo_summary([1.0, 0.5, 0.5, 0.0])
    se = math.sqrt(1 / 24)
    assert r["score"] == 0.5 and r["elo"] == 0.0 and r["pairs"] == 4
    assert r["score_se"] == pytest.approx(se)
    lo = 0.5 - 1.959963984540054 * se  # 0.09993
    assert r["elo_ci"][0] == pytest.approx(-400 * math.log10(1 / lo - 1)) and r["elo_ci"][0] == pytest.approx(-381.8, abs=0.1)
    assert r["elo_ci"][1] == pytest.approx(-r["elo_ci"][0])
    # pairs (1, 1/2, 1, 1/2): mean 3/4, sample variance 4 (1/4)^2 / 3 = 1/12, standard error sqrt(1/48)
    r = elo_summary([1.0, 0.5, 1.0, 0.5])
    se = math.sqrt(1 / 48)
    assert r["score"] == 0.75 and r["score_se"] == pytest.approx(se)
    assert r["elo"] == pytest.approx(190.849, abs=1e-3)
    assert r["elo_ci"][0] == pytest.approx(-400 * math.log10(1 / (0.75 - 1.959963984540054 * se) - 1))
    assert r["elo_ci"][1] == math.inf  # the upper end of the score interval passes 1


def test_elo_interval_all_draws_and_a_clean_sweep():
    from betazero_b200.match import elo_summary

    r = elo_summary([0.5] * 100)
    assert r["score"] == 0.5 and r["elo"] == 0.0 and r["elo_ci"] == [0.0, 0.0] and r["score_se"] == 0.0
    r = elo_summary([1.0] * 10)
    assert r["score"] == 1.0 and r["elo"] == math.inf and r["elo_ci"] == [math.inf, math.inf]
    r = elo_summary([0.0] * 10)
    assert r["elo"] == -math.inf and r["elo_ci"] == [-math.inf, -math.inf]
    r = elo_summary([0.25])  # one pair: no spread to estimate
    assert r["score_se"] == 0.0 and r["elo_ci"][0] == r["elo_ci"][1] == r["elo"]
    assert math.isnan(elo_summary([])["score"])


def test_match_refuses_odd_game_counts_before_touching_a_device():
    from betazero_b200.match import BatchedMatch

    with pytest.raises(ValueError, match="even"):
        BatchedMatch(None, None, 7, 16)
    with pytest.raises(ValueError, match="n_leaves"):
        BatchedMatch(None, None, 8, 12, n_leaves=3)
