"""Host side of head-to-head evaluation: the board -> (class, suit permutation) deal map of Flop5Holdem, the lexicographic
board rank the kernel uses, the counter uniforms, the C struct mirror of prl_h2h_t and the public import paths."""
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _flop5_spec_and_map():
    from pokerrl_b200.game import games
    from pokerrl_b200.game.holdem_boards import BoardSpec, board_class_map
    spec = BoardSpec.full_game(games.Flop5Holdem.RULES)
    return spec, board_class_map(spec)


def test_every_board_maps_onto_its_class_representative():
    from itertools import permutations
    from pokerrl_b200.game.holdem_boards import _combos_52_5
    spec, (cls, perm) = _flop5_spec_and_map()
    boards = _combos_52_5().astype(np.int64)
    perms = np.array(list(permutations(range(4))))[perm]  # [n_boards, 4]: suit -> suit
    mapped = np.sort((boards // 4) * 4 + np.take_along_axis(perms, boards % 4, axis=1), axis=1)
    assert np.array_equal(mapped, spec.boards[cls].astype(np.int64))
    assert np.bincount(cls, minlength=spec.boards.shape[0]).tolist() == (spec.board_mult * 24).round().astype(int).tolist()


def test_hand_on_the_board_keeps_its_strength_on_the_representative():
    """the direction of s: hand h on the dealt board ranks exactly like hand sym_perm[s][h] on the class representative
    (all 1326 hands on 3000 boards, strengths from the C hand evaluator oracle)"""
    from twocard_common import oracle_ranks
    from pokerrl_b200.game.holdem_boards import _combos_52_5
    spec, (cls, perm) = _flop5_spec_and_map()
    boards = _combos_52_5()
    pick = np.random.default_rng(5).choice(boards.shape[0], 3000, replace=False)
    dealt, rep = oracle_ranks(boards[pick]), oracle_ranks(spec.boards[cls[pick]])
    c1, c2 = np.triu_indices(52, k=1)
    for k, b in enumerate(pick):
        free = ~(np.isin(c1, boards[b]) | np.isin(c2, boards[b]))
        hp = spec.sym_perm[perm[b]].astype(np.int64)
        assert np.array_equal(dealt[k][free], rep[k][hp][free]), b


def test_lexicographic_board_rank_equals_the_enumeration_order():
    from math import comb
    from pokerrl_b200.cfr.TabularCFREvalAgent import _lex_rank_52_5
    from pokerrl_b200.game.holdem_boards import _combos_52_5
    boards = _combos_52_5().astype(np.int64)
    colex = sum(np.array([comb(51 - c, 5 - i) for c in range(52)], np.int64)[boards[:, i]] for i in range(5))
    assert np.array_equal(comb(52, 5) - 1 - colex, np.arange(boards.shape[0]))
    for r in (0, 1, 777, 1234567, boards.shape[0] - 1):
        assert _lex_rank_52_5(boards[r]) == r


def test_counter_uniforms_are_deterministic_and_in_the_unit_interval():
    from pokerrl_b200.eval.head_to_head.match import counter_uniforms
    u = counter_uniforms(7, np.arange(1000), 12)
    assert u.shape == (1000, 12) and u.min() >= 0.0 and u.max() < 1.0
    assert np.array_equal(u[500:], counter_uniforms(7, np.arange(500, 1000), 12))
    assert not np.array_equal(u, counter_uniforms(8, np.arange(1000), 12))
    assert abs(u.mean() - 0.5) < 0.01


def test_h2h_struct_mirror_matches_the_header(tmp_path):
    from pokerrl_b200 import _native
    cls = _native.PrlH2H
    src = ['#include <stdio.h>', '#include <stddef.h>', '#include "pokerrl_b200.h"', 'int main(void) {',
           'printf("size %zu\\n", sizeof(prl_h2h_t));']
    for f, _ in cls._fields_:
        src.append('printf("%s %%zu\\n", offsetof(prl_h2h_t, %s));' % (f, f))
    src.append("return 0; }")
    c_file, exe = tmp_path / "h2h.c", tmp_path / "h2h"
    c_file.write_text("\n".join(src))
    subprocess.check_call(["/usr/bin/gcc", "-I", os.path.join(ROOT, "include"), str(c_file), "-o", str(exe)])
    got = dict(line.split() for line in subprocess.check_output([str(exe)], text=True).splitlines())
    import ctypes as C
    assert int(got["size"]) == C.sizeof(cls)
    for f, _ in cls._fields_:
        assert int(got[f]) == getattr(cls, f).offset, f


def test_h2h_args_and_compat_imports_resolve():
    from pokerrl_b200.eval.head_to_head import H2HArgs
    a = H2HArgs(n_hands=10)
    assert a.n_hands == 10 and a.batch_size == 1 << 20 and a.seed == 0
    code = ("from PokerRL.eval.head_to_head.LocalHead2HeadMaster import LocalHead2HeadMaster\n"
            "from PokerRL.eval.head_to_head.H2HArgs import H2HArgs\n"
            "from pokerrl_b200.eval.head_to_head import LocalHead2HeadMaster as native\n"
            "assert LocalHead2HeadMaster is native and H2HArgs(5).n_hands == 5\n"
            "print('ok')\n")
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([os.path.join(ROOT, "pokerrl_b200", "compat"), ROOT]))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr


def test_fixture_exact_leduc_values_agree_with_an_independent_enumeration():
    """the exact match values the fixture generator enumerated through the reference's PokerEnv equal a float64 walk of this
    package's flat tree over every deal, with the policies restated in tests/h2h_common.py"""
    from h2h_common import exact_one_card
    from pokerrl_b200.game import bet_sets, games
    gold = np.load(os.path.join(ROOT, "tests", "golden", "h2h_runs.npz"))
    for game, bet_set in ((games.StandardLeduc, bet_sets.POT_ONLY), (games.DiscretizedNLLeduc, bet_sets.B_3)):
        args = game.ARGS_CLS(n_seats=2, starting_stack_sizes_list=[game.DEFAULT_STACK_SIZE] * 2,
                             bet_sizes_list_as_frac_of_pot=list(bet_set))
        got, want = exact_one_card(game, args), gold[game.__name__ + "_exact"]
        err = np.abs(got - want).max() / np.abs(want).max()
        print("%s: exact %s, reference enumeration %s, rel. error %.1e" % (game.__name__, got, want, err))
        assert err <= 1e-9
