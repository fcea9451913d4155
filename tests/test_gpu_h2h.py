"""Head-to-head matches on the GPU (eval/head_to_head, csrc/h2h.cu): the device path against the per-hand host loop on the
same deals and uniforms, sampled means against the exact match value, batch independence, the master's logged series,
and the tabular agent of a full-game Flop5Holdem board-engine solver playing matches and LBR."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _t_prof(game, bet_set, stacks=None, modes=("AVG",)):
    from pokerrl_b200.rl.base_cls.TrainingProfileBase import TrainingProfileBase
    return TrainingProfileBase("h2h", game, list(bet_set), eval_stack_sizes=stacks, eval_modes_of_algo=modes)


def _cfr_agent(game, bet_set, iters, stack=None):
    from pokerrl_b200.cfr.CFRPlus import CFRPlus
    from pokerrl_b200.cfr.TabularCFREvalAgent import TabularCFREvalAgent
    from pokerrl_b200.rl.base_cls.workers.ChiefBase import ChiefBase
    cfr = CFRPlus(name="h", chief_handle=ChiefBase(None), game_cls=game, agent_bet_set=list(bet_set), delay=0,
                  starting_stack_sizes=None if stack is None else [stack])
    for _ in range(iters):
        cfr.iteration()
    stacks = None if stack is None else [[stack, stack]]
    agent = TabularCFREvalAgent.from_cfr(_t_prof(game, bet_set, stacks), cfr)
    del cfr
    torch.cuda.empty_cache()
    return agent


def _uniform_agent(like):
    """a tabular agent on `like`'s tree that plays every legal action with the same probability"""
    from pokerrl_b200.cfr.TabularCFREvalAgent import TabularCFREvalAgent
    ft, fp = like.own_tree()
    inv = 1.0 / ft.n_children[ft.parent[np.nonzero(ft.slot >= 0)[0]]].astype(np.float32)
    agent = TabularCFREvalAgent(t_prof=like.t_prof)
    if isinstance(like._table, torch.Tensor):
        tab = torch.from_numpy(inv).cuda()[:, None].expand(-1, like._table.shape[1]).contiguous()
    else:
        tab = np.repeat(inv[:, None], ft.R, axis=1)
    agent.update_weights((tab, fp))
    agent.set_stack_size(like._stack_size)
    return agent


def _replay_host_vs_device(a, b, stack, n_per_seat, n_device, seed=11):
    """device hands [0, n) and [N, N + n) of a match of N = n_device hands per seat, replayed through the host loop"""
    from pokerrl_b200.eval.head_to_head.match import counter_uniforms, deal, play_match_details
    dev = play_match_details(a, b, n_device, stack, seed=seed, winnings=True)
    ids = np.concatenate([np.arange(n_per_seat), n_device + np.arange(n_per_seat)])
    decks = np.concatenate([deal(a.env_bldr, stack, seed, 0, n_per_seat), deal(a.env_bldr, stack, seed, n_device, n_per_seat)])
    u = counter_uniforms(seed, ids, 64)
    host = play_match_details(a, b, n_per_seat, stack, decks=decks, uniforms=u, host_loop=True)
    want = dev["winnings"][ids]
    err = np.abs(host["winnings"] - want).max() / max(1.0, np.abs(want).max())
    # the same deals and uniforms through the device path's replay inputs give the same hands as well
    again = play_match_details(a, b, n_per_seat, stack, decks=decks, uniforms=u, winnings=True)
    assert np.array_equal(again["winnings"], want)
    return dev, err


@pytest.mark.parametrize("game_name", ["StandardLeduc", "DiscretizedNLLeduc"])
def test_leduc_device_host_exact(game_name):
    from pokerrl_b200.eval.head_to_head.match import exact_head_to_head, play_match_details
    from pokerrl_b200.game import bet_sets, games
    game = getattr(games, game_name)
    bet_set = bet_sets.B_3 if game_name == "DiscretizedNLLeduc" else bet_sets.POT_ONLY
    a = _cfr_agent(game, bet_set, 100)
    b = _uniform_agent(a)
    stack = [game.DEFAULT_STACK_SIZE] * 2
    dev, err = _replay_host_vs_device(a, b, stack, 500, 1 << 16)
    assert err <= 1e-6, err
    exact = exact_head_to_head(a, b, stack)
    big = play_match_details(a, b, 1 << 23, stack, seed=5)
    print("%s: CFR+ (100 it) vs uniform: exact %.3f, sampled %.3f +- %.3f mbb/g over %d hands; host replay err %.1e"
          % (game_name, exact, big["mean"], big["half_width"], big["n"], err))
    assert abs(big["mean"] - exact) <= 4 * big["half_width"]


def test_batch_size_does_not_change_the_result():
    from pokerrl_b200.eval.head_to_head.match import play_match_details
    from pokerrl_b200.game import bet_sets, games
    a = _cfr_agent(games.DiscretizedNLLeduc, bet_sets.B_3, 10)
    b = _uniform_agent(a)
    stack = [games.DiscretizedNLLeduc.DEFAULT_STACK_SIZE] * 2
    r = [play_match_details(a, b, 1 << 19, stack, seed=3, batch_size=bs, winnings=True) for bs in (1 << 16, 1 << 20)]
    assert r[0]["sum"] == r[1]["sum"] and r[0]["sum_sq"] == r[1]["sum_sq"]
    assert np.array_equal(r[0]["winnings"], r[1]["winnings"])


def test_flop5_push_fold_sampled_equals_exact():
    from pokerrl_b200.eval.head_to_head.match import exact_head_to_head, play_match_details
    from pokerrl_b200.game import games
    g = games.Flop5Holdem
    a, b = _cfr_agent(g, [1.0], 30, stack=300), _cfr_agent(g, [1.0], 2, stack=300)
    stack = [300, 300]
    dev, err = _replay_host_vs_device(a, b, stack, 300, 1 << 16)
    assert err <= 1e-6, err
    exact = exact_head_to_head(a, b, stack)
    big = play_match_details(a, b, 1 << 23, stack, seed=9)
    print("Flop5 push/fold: CFR+ 30 it vs 2 it: exact %.3f, sampled %.3f +- %.3f mbb/g; host replay err %.1e"
          % (exact, big["mean"], big["half_width"], err))
    assert abs(big["mean"] - exact) <= 4 * big["half_width"]


def test_master_logs_per_stack_and_multi_stack_series():
    from pokerrl_b200.cfr.TabularCFREvalAgent import TabularCFREvalAgent
    from pokerrl_b200.eval.head_to_head import H2HArgs, LocalHead2HeadMaster
    from pokerrl_b200.game import bet_sets, games
    from pokerrl_b200.rl.base_cls.workers.ChiefBase import ChiefBase
    game = games.StandardLeduc
    a = _cfr_agent(game, bet_sets.POT_ONLY, 20)
    t_prof = _t_prof(game, bet_sets.POT_ONLY, stacks=[[13, 13], [13, 13]])
    t_prof.module_args["h2h"] = H2HArgs(n_hands=1 << 16, seed=1)
    chief = ChiefBase(t_prof=None)
    w = (a._table, a._fingerprint)
    chief.pull_current_eval_strategy = lambda info: (w, info)
    m = LocalHead2HeadMaster(t_prof=t_prof, chief_handle=chief, eval_agent_cls=TabularCFREvalAgent)
    m.set_modes(["AVG", "AVG"])
    m.update_weights()
    m.evaluate(iter_nr=4)
    exps, gname = chief.get_experiments(), "Evaluation/" + game.WIN_METRIC
    for s in ("Total", "Conf_lower95", "Conf_upper95"):
        assert exps["h2h AVG_stack_13: Head2Head_Winnings " + s][gname][0][0] == 4
    tot = exps["h2h Head2HeadMulti_Stack: Head2Head_Winnings Averaged Total"][gname]
    lo = exps["h2h Head2Head: Head2Head_Winnings Conf_lower95"][gname]
    hi = exps["h2h Head2Head: Head2Head_Winnings Conf_upper95"][gname]
    assert lo[0][1] <= tot[0][1] <= hi[0][1]
    print("master: self-play %.3f [%.3f, %.3f] mbb/g" % (tot[0][1], lo[0][1], hi[0][1]))


@pytest.fixture(scope="module")
def flop5_agent():
    from pokerrl_b200.game import games
    a = _cfr_agent(games.Flop5Holdem, [1.0], 3)
    torch.cuda.synchronize()
    print("Flop5Holdem board-engine agent built; max memory allocated %.1f GB" % (torch.cuda.max_memory_allocated() / 1e9))
    return a


def test_full_game_flop5_matches_on_device_and_host(flop5_agent):
    a = flop5_agent
    b = _uniform_agent(a)
    stack = [20000, 20000]
    dev, err = _replay_host_vs_device(a, b, stack, 1000, 1 << 19)
    print("Flop5Holdem full game, CFR+ (3 it) vs uniform: %.1f +- %.1f mbb/g over %d hands; host replay of 2000 hands err %.1e; "
          "max memory allocated %.1f GB" % (dev["mean"], dev["half_width"], dev["n"], err, torch.cuda.max_memory_allocated() / 1e9))
    assert dev["desync"] == 0 and err <= 1e-6
    del b
    torch.cuda.empty_cache()


def test_lbr_runs_against_the_full_game_tabular_agent(flop5_agent):
    from pokerrl_b200.cfr.TabularCFREvalAgent import TabularCFREvalAgent
    from pokerrl_b200.eval.lbr.LBRArgs import LBRArgs
    from pokerrl_b200.eval.lbr.LocalLBRWorker import LocalLBRWorker
    from pokerrl_b200.game import games
    from pokerrl_b200.game.Poker import Poker
    t_prof = _t_prof(games.Flop5Holdem, [1.0], stacks=[[20000, 20000]])
    t_prof.module_args["lbr"] = LBRArgs(n_lbr_hands_per_seat=4, lbr_check_to_round=Poker.FLOP)
    w = LocalLBRWorker(t_prof=t_prof, chief_handle=None, eval_agent_cls=TabularCFREvalAgent)
    w.update_weights((flop5_agent._table, flop5_agent._fingerprint))
    np.random.seed(0)
    out = [w.run(seat, 4, "AVG", [20000, 20000]) for seat in (0, 1)]
    assert all(o is not None and o.shape == (4,) and np.isfinite(o).all() for o in out)
    print("LBR vs Flop5Holdem CFR+ agent: winnings", np.concatenate(out))
