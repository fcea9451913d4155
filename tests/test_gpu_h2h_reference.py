"""Head-to-head against the REFERENCE (tests/golden/h2h_runs.npz, produced by running PokerRL's own
LocalHead2HeadMaster._run_eval between two fixed policies: oracle/gen_golden_h2h.py): the recorded hands replayed through the
host loop and the device path with the recorded deals and uniforms win the recorded chips hand for hand, and the exact match
value of both Leduc games equals the reference's float64 enumeration.  Also the board-engine average strategy table against
a host restatement of its normalisation."""
import os

import numpy as np
import pytest

from h2h_common import policy_agent

pytestmark = pytest.mark.gpu
GOLD = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "h2h_runs.npz"))


def _game(name):
    from pokerrl_b200.game import bet_sets, games
    from pokerrl_b200.rl.base_cls.TrainingProfileBase import TrainingProfileBase
    game = getattr(games, name)
    bet_set = bet_sets.B_3 if name == "DiscretizedNLLeduc" else bet_sets.POT_ONLY
    stack = [game.DEFAULT_STACK_SIZE] * 2
    return game, TrainingProfileBase("h2h", game, list(bet_set), eval_stack_sizes=[stack]), stack


@pytest.mark.parametrize("name", ["StandardLeduc", "DiscretizedNLLeduc", "Flop5Holdem"])
def test_reference_matches_replay_on_both_paths(name):
    import torch
    from pokerrl_b200.eval.head_to_head.match import play_match_details
    game, t_prof, stack = _game(name)
    a, b = policy_agent(t_prof, "A", stack), policy_agent(t_prof, "B", stack)
    decks, u, want = GOLD[name + "_decks"], GOLD[name + "_uniforms"], GOLD[name + "_winnings"]
    n = want.size // 2
    host = play_match_details(a, b, n, stack, decks=decks, uniforms=u, host_loop=True)
    dev = play_match_details(a, b, n, stack, decks=decks, uniforms=u, winnings=True)
    scale = max(1.0, float(np.abs(want).max()))
    e_host = float(np.abs(host["winnings"] - want).max()) / scale
    e_dev = float(np.abs(dev["winnings"] - want).max()) / scale
    print("%s: %d reference hands, host loop err %.1e, device path err %.1e, desync %d, mean %.2f (reference %.2f) mbb/g"
          % (name, want.size, e_host, e_dev, dev["desync"], dev["mean"], float(want.astype(np.float64).mean())))
    assert dev["desync"] == 0 and e_host <= 1e-6 and e_dev <= 1e-6
    del a, b
    torch.cuda.empty_cache()


@pytest.mark.parametrize("name", ["StandardLeduc", "DiscretizedNLLeduc"])
def test_exact_value_equals_the_reference_enumeration(name):
    from pokerrl_b200.eval.head_to_head.match import exact_head_to_head
    game, t_prof, stack = _game(name)
    a, b = policy_agent(t_prof, "A", stack), policy_agent(t_prof, "B", stack)
    got, want = exact_head_to_head(a, b, stack), float(GOLD[name + "_exact"][2])
    err = abs(got - want) / abs(want)
    print("%s: exact_head_to_head %.9f, reference enumeration %.9f, rel. error %.1e" % (name, got, want, err))
    assert err <= 1e-6


@pytest.mark.parametrize("algo,iters", [("CFRPlus", 1), ("CFRPlus", 3), ("LinearCFR", 2), ("VanillaCFR", 2)])
def test_board_strategy_table_normalises_like_the_level_engine(algo, iters):
    """CFR+ at iteration delay + 1: regret matching of the regret rows; later: the average as is; Vanilla / Linear: the
    reach-weighted sums normalised per decision node, uniform where they are 0 - on a 32-board Flop5Holdem instance"""
    from twocard_common import fhp_tree, random_board_spec
    from pokerrl_b200.board_engine import BoardCFRSolver
    from pokerrl_b200.cfr.TabularCFREvalAgent import board_strategy_table
    from pokerrl_b200.game import games
    spec = random_board_spec(32, 7)
    ft = fhp_tree(spec)
    g = games.Flop5Holdem
    args = g.ARGS_CLS(n_seats=2, starting_stack_sizes_list=[20000, 20000], bet_sizes_list_as_frac_of_pot=[1.0])
    s = BoardCFRSolver(g, args, spec, algo=algo)
    s.iteration(iters)
    regret, avg = (t.cpu().numpy()[:, :ft.R].astype(np.float32) for t in s.natural_tables(ft))
    got = board_strategy_table(s, ft).cpu().numpy()[:, :ft.R]
    if algo == "CFRPlus" and iters > 1:
        want = avg
    else:
        src = np.maximum(regret, 0) if algo == "CFRPlus" else avg
        want = np.empty_like(src)
        for n in np.nonzero((ft.kind <= 1) & (ft.first_child >= 0))[0]:
            a, fs = ft.n_children[n], ft.first_slot[n]
            tot = src[fs:fs + a].sum(axis=0, keepdims=True)
            with np.errstate(divide="ignore", invalid="ignore"):
                want[fs:fs + a] = np.where(tot == 0, np.float32(1.0 / a), src[fs:fs + a] / tot)
    err = float(np.abs(got - want).max())
    print("%s after %d iterations: board_strategy_table vs host normalisation, max abs diff %.1e" % (algo, iters, err))
    assert err <= 1e-6
