"""Golden HEAD-TO-HEAD matches, produced by RUNNING THE REFERENCE's LocalHead2HeadMaster._run_eval
(PokerRL/eval/head_to_head/LocalHead2HeadMaster.py:81-126) between two modes of an agent with fixed policies, plus the exact
value of the Leduc matches by enumerating every deal and action path through the reference's PokerEnv (TEST
INFRASTRUCTURE; needs /root/reference):

    python oracle/gen_golden_h2h.py      # writes tests/golden/h2h_runs.npz

Games: StandardLeduc, DiscretizedNLLeduc (bet_sets.B_3), Flop5Holdem.  Mode "A" and mode "B" play different policies, each a
function of (the hand's suit-invariant class, the legal actions, the street) only, so that a table over suit-isomorphism
classes represents them; the policy is restated in tests/h2h_common.py.  Recorded per hand: the deal (hole cards + the rest of
the deck in drawing order), the uniforms both agents drew in decision order, agent 0's (mode A's) winnings.  Hands [0, n)
have mode A in seat 0, hands [n, 2n) in seat 1."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import ref_harness as rh  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
N_HANDS = {"StandardLeduc": 200, "DiscretizedNLLeduc": 150, "Flop5Holdem": 100}
POLICY = {"A": (7, 13, 3, 5), "B": (5, 3, 11, 7)}  # weight 1 + ((c0 * class + c1 * action + c2 * street) mod m)


def hand_classes(n_cards, n_hole, n_suits):
    """int64 [R]: one-card games the card's rank; two-card games (low rank, high rank, suited)"""
    if n_hole == 1:
        return np.arange(n_cards, dtype=np.int64) // n_suits
    c1, c2 = np.triu_indices(n_cards, k=1)
    r1, r2 = c1 // n_suits, c2 // n_suits
    return (np.minimum(r1, r2) * 13 + np.maximum(r1, r2)) * 2 + (c1 % n_suits == c2 % n_suits)


def policy_table(mode, classes, n_actions, legal, street):
    c0, c1, c2, m = POLICY[mode]
    a = np.arange(n_actions, dtype=np.int64)[None, :]
    w = (1 + ((c0 * classes[:, None] + c1 * a + c2 * street) % m)).astype(np.float32)
    mask = np.zeros(n_actions, np.float32)
    mask[list(legal)] = 1.0
    w = w * mask[None, :]
    return (w / w.sum(axis=1, keepdims=True)).astype(np.float32)


def main():
    rh.import_reference()
    M = sys.modules.get("PokerRL.eval.head_to_head.LocalHead2HeadMaster")
    if M is None:
        import importlib
        importlib.import_module("PokerRL.eval.head_to_head.LocalHead2HeadMaster")
        M = sys.modules["PokerRL.eval.head_to_head.LocalHead2HeadMaster"]
    from PokerRL.eval.head_to_head.H2HArgs import H2HArgs
    from PokerRL.game import bet_sets, games
    from PokerRL.rl.base_cls.EvalAgentBase import EvalAgentBase

    rec = {"draws": None, "decks": []}

    class PolicyAgent(EvalAgentBase):
        ALL_MODES = ["A", "B"]

        def can_compute_mode(self):
            return True

        def update_weights(self, w):
            pass

        def _state_dict(self):
            return {}

        def _load_state_dict(self, s):
            pass

        def get_a_probs_for_each_hand(self):
            env = self._internal_env_wrapper.env
            r = self.env_bldr.rules
            return policy_table(self._mode, hand_classes(r.N_CARDS_IN_DECK, r.N_HOLE_CARDS, r.N_SUITS), self.env_bldr.N_ACTIONS,
                                env.get_legal_actions(), env.current_round)

        def get_action(self, step_env=True, need_probs=False):  # EvalAgentBase.get_action as the project restates it
            env = self._internal_env_wrapper.env
            probs = self.get_a_probs_for_each_hand()
            row = probs[env.get_range_idx(p_id=env.current_player.seat_id)].astype(np.float64)
            u = float(np.random.random())
            rec["draws"].append(u)
            action = int(min(np.searchsorted(np.cumsum(row), u, side="right"), row.size - 1))
            while row[action] == 0 and action > 0:
                action -= 1
            if step_env:
                self._internal_env_wrapper.step(action=action)
            return action, (probs if need_probs else None)

        def reset(self, deck_state_dict=None):
            if self is agents[0]:  # once per hand: the deal of the table
                lut = self.env_bldr.lut_holder
                hands = np.concatenate([np.asarray(lut.get_1d_cards(np.asarray(h))).reshape(-1) for h in deck_state_dict["hand"]])
                rest = np.asarray(lut.get_1d_cards(np.asarray(deck_state_dict["deck"]["deck_remaining"]))).reshape(-1)
                rec["decks"].append(np.concatenate([hands, rest]).astype(np.int8))
                rec["draws"] = []
                rec["all_draws"].append(rec["draws"])
            super().reset(deck_state_dict=deck_state_dict)

    class Chief:
        def create_experiment(self, name):
            return name

        def add_scalar(self, *a):
            pass

    out = {}
    agents = []
    for game, bet_set in ((games.StandardLeduc, bet_sets.POT_ONLY), (games.DiscretizedNLLeduc, bet_sets.B_3),
                          (games.Flop5Holdem, bet_sets.POT_ONLY)):
        name = game.__name__
        stack = [game.DEFAULT_STACK_SIZE] * 2
        env_args = game.ARGS_CLS(n_seats=2, starting_stack_sizes_list=list(stack), bet_sizes_list_as_frac_of_pot=list(bet_set))

        class TProf:
            n_seats = 2
            DISTRIBUTED = CLUSTER = DEBUGGING = HAVE_GPU = False
            env_builder_cls_str = "VanillaEnvBuilder"
            game_cls_str = name
            device_inference = None
            eval_modes_of_algo = ["A"]
            eval_stack_sizes = [list(stack)]
            module_args = {"env": env_args, "h2h": H2HArgs(n_hands=N_HANDS[name])}
        TProf.name = "h2h"

        master = M.LocalHead2HeadMaster(t_prof=TProf(), chief_handle=Chief(), eval_agent_cls=PolicyAgent)
        agents[:] = master._eval_agents
        master.set_modes(["A", "B"])
        for e in agents:
            e.set_stack_size(list(stack))
        rec["decks"], rec["all_draws"] = [], []
        got = {}

        def keep_winnings(scores, got=got):  # the per-hand array _run_eval hands to the interval
            got["w"] = np.array(scores)
            return 0.0, 0.0
        master._get_95confidence = keep_winnings
        np.random.seed(4321)
        master._run_eval(stack_size=list(stack))
        n = 2 * N_HANDS[name]
        assert len(rec["decks"]) == n and all(len(set(d.tolist())) == d.size for d in rec["decks"])
        k = max(len(d) for d in rec["all_draws"])
        draws = np.full((n, k), -1.0)
        for i, d in enumerate(rec["all_draws"]):
            draws[i, :len(d)] = d
        out[name + "_decks"] = np.array(rec["decks"], np.int8)
        out[name + "_uniforms"] = draws
        out[name + "_winnings"] = got["w"].astype(np.float32)
        print(name, "hands", n, "mean winnings of mode A per seat", got["w"][:n // 2].mean(), got["w"][n // 2:].mean(),
              "max decisions", k)
        if game.RULES.N_HOLE_CARDS == 1:
            out[name + "_exact"] = np.array(exact_value(game, env_args, stack, master._eval_env_bldr))
            print(name, "exact value of mode A per seat and averaged", out[name + "_exact"])
    np.savez_compressed(os.path.join(OUT, "h2h_runs.npz"), **out)
    print("wrote h2h_runs.npz")


def exact_value(game, env_args, stack, env_bldr):
    """float64 [3]: mode A's expected winnings per hand with A in seat 0, in seat 1, and their average - every ordered deal
    (hole cards, board card) with equal probability, every action path through the reference's PokerEnv weighted by the
    policies' float32 probabilities in float64 (one process per (seat, first hole card); sums in deal order)"""
    import multiprocessing as mp
    _JOB.update(game=game, stack=stack, env_bldr=env_bldr)
    n_cards = game.RULES.N_CARDS_IN_DECK
    with mp.get_context("fork").Pool(min(8, 2 * n_cards)) as pool:
        parts = pool.map(_deals_of, [(seat_a, c0) for seat_a in (0, 1) for c0 in range(n_cards)])
    vals = []
    for seat_a in (0, 1):
        tot, n = 0.0, 0
        for (s_a, _), (t, k) in zip([(sa, c) for sa in (0, 1) for c in range(n_cards)], parts):
            if s_a == seat_a:
                tot += t
                n += k
        vals.append(tot / n)
    return [vals[0], vals[1], 0.5 * (vals[0] + vals[1])]


_JOB = {}


def _deals_of(job):
    seat_a, c0 = job
    game, stack, env_bldr = _JOB["game"], _JOB["stack"], _JOB["env_bldr"]
    env = env_bldr.get_new_env(is_evaluating=True, stack_size=list(stack))
    r = game.RULES
    classes = hand_classes(r.N_CARDS_IN_DECK, r.N_HOLE_CARDS, r.N_SUITS)
    lut = env_bldr.lut_holder
    n_cards = r.N_CARDS_IN_DECK
    tot, n_deals = 0.0, 0
    for c1 in range(n_cards):
        if c1 == c0:
            continue
        rest = [c for c in range(n_cards) if c not in (c0, c1)]
        for b in range(len(rest)):
            order = [rest[b]] + rest[:b] + rest[b + 1:]
            env.reset()
            csd = env.cards_state_dict()  # the reference's layout, then this deal's cards
            csd["hand"] = [lut.get_2d_cards(np.array([c0], np.int8)), lut.get_2d_cards(np.array([c1], np.int8))]
            csd["deck"]["deck_remaining"] = lut.get_2d_cards(np.array(order, np.int8))
            env.reset(deck_state_dict=csd)
            tot += _walk(env, seat_a, classes, env_bldr.N_ACTIONS, (c0, c1))
            n_deals += 1
    return tot, n_deals


def _walk(env, seat_a, classes, n_actions, hole):
    p = env.current_player.seat_id
    legal = env.get_legal_actions()
    probs = policy_table("A" if p == seat_a else "B", classes, n_actions, legal, env.current_round)[hole[p]]
    sd = env.state_dict()
    v = 0.0
    for a in legal:
        env.load_state_dict(sd)
        _, r, done, _ = env.step(a)
        w = float(probs[a])
        v += w * (r[seat_a] * env.REWARD_SCALAR * env.EV_NORMALIZER if done else _walk(env, seat_a, classes, n_actions, hole))
    env.load_state_dict(sd)
    return v


if __name__ == "__main__":
    main()
