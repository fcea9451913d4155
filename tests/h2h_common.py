"""Helpers of the head-to-head fixture tests: the two fixed policies the fixture generator (oracle/gen_golden_h2h.py) gave the
REFERENCE's LocalHead2HeadMaster, as tabular agents of this package, and an exact match value computed on this package's flat
tree in float64 (independent of the reference's env)."""
import numpy as np

POLICY = {"A": (7, 13, 3, 5), "B": (5, 3, 11, 7)}  # weight 1 + ((c0 * class + c1 * action + c2 * street) mod m)


def hand_classes(n_cards, n_hole, n_suits):
    """int64 [R]: one-card games the card's rank; two-card games (low rank, high rank, suited) - invariant under suit
    permutations, so that a table over suit-isomorphism classes of boards represents the policy"""
    if n_hole == 1:
        return np.arange(n_cards, dtype=np.int64) // n_suits
    c1, c2 = np.triu_indices(n_cards, k=1)
    r1, r2 = c1 // n_suits, c2 // n_suits
    return (np.minimum(r1, r2) * 13 + np.maximum(r1, r2)) * 2 + (c1 % n_suits == c2 % n_suits)


def policy_table(mode, classes, n_actions, legal, street):
    """float32 [R, N_ACTIONS]: the policy's weights on the legal actions, rows normalised"""
    c0, c1, c2, m = POLICY[mode]
    a = np.arange(n_actions, dtype=np.int64)[None, :]
    w = (1 + ((c0 * classes[:, None] + c1 * a + c2 * street) % m)).astype(np.float32)
    mask = np.zeros(n_actions, np.float32)
    mask[list(legal)] = 1.0
    w = w * mask[None, :]
    return (w / w.sum(axis=1, keepdims=True)).astype(np.float32)


def policy_agent(t_prof, mode, stack, device="cuda"):
    """TabularCFREvalAgent whose table plays `mode` on the flat tree of `stack` (device table, built in slices)"""
    import torch
    from pokerrl_b200.cfr.TabularCFREvalAgent import TabularCFREvalAgent
    agent = TabularCFREvalAgent(t_prof=t_prof)
    agent.set_stack_size(stack)
    ft, fp = agent.own_tree()  # no table yet: no fingerprint to check
    r = ft.rules
    c0, c1, c2, m = POLICY[mode]
    cls = torch.from_numpy(hand_classes(r.N_CARDS_IN_DECK, r.N_HOLE_CARDS, r.N_SUITS)).to(device)
    child = np.nonzero(ft.slot >= 0)[0]  # flat order == slot order
    par = ft.parent[child]
    act = torch.from_numpy(ft.action[child].astype(np.int64)).to(device)
    street = torch.from_numpy(ft.round[par].astype(np.int64)).to(device)
    dec = np.nonzero((ft.kind <= 1) & (ft.first_child >= 0))[0]
    dec_idx = np.full(ft.n_nodes, -1, np.int64)
    dec_idx[dec] = np.arange(dec.size)
    seg = torch.from_numpy(dec_idx[par]).to(device)
    tab = torch.empty((child.size, ft.R), dtype=torch.float32, device=device)
    CH = 1 << 16
    for i in range(0, child.size, CH):
        tab[i:i + CH] = (1 + (c0 * cls[None, :] + c1 * act[i:i + CH, None] + c2 * street[i:i + CH, None]) % m).float()
    tot = torch.zeros((dec.size, ft.R), dtype=torch.float32, device=device)
    tot.index_add_(0, seg, tab)
    for i in range(0, child.size, CH):
        tab[i:i + CH] /= tot[seg[i:i + CH]]
    agent.update_weights((tab if device != "cpu" else tab.numpy(), fp))
    return agent


def exact_one_card(game, env_args):
    """float64 [3]: mode A's expected winnings (game EV unit) against mode B with A in seat 0, in seat 1, and their average,
    by walking this package's flat tree for every ordered deal (hole cards, board card) of a one-card game"""
    from pokerrl_b200.game.flat_tree import FlatTree, KIND_CHANCE, KIND_FOLD
    ft = FlatTree(game, env_args)
    r = game.RULES
    classes = hand_classes(r.N_CARDS_IN_DECK, 1, r.N_SUITS)
    n_act = env_args.N_ACTIONS
    start = np.asarray(env_args.starting_stack_sizes_list, np.int64)
    n_cards = r.N_CARDS_IN_DECK

    def strength(c, b):
        return r.PAIR_BONUS + c // r.N_SUITS if c // r.N_SUITS == b // r.N_SUITS else c // r.N_SUITS

    cache = {}

    def walk(n, seat_a, hole, b):
        k = ft.kind[n]
        if k <= 1:
            fc, a = ft.first_child[n], ft.n_children[n]
            legal = ft.action[fc:fc + a]
            key = ("A" if k == seat_a else "B", tuple(legal.tolist()), int(ft.round[n]))
            if key not in cache:
                cache[key] = policy_table(key[0], classes, n_act, key[1], key[2])
            probs = cache[key][hole[k]]
            return sum(float(probs[legal[j]]) * walk(fc + j, seat_a, hole, b) for j in range(a))
        if k == KIND_CHANCE:
            return walk(ft.first_child[n] + b, seat_a, hole, b)  # one board card: the j-th child is card j
        put = start - ft.stack[n]
        if k == KIND_FOLD:
            folder = int(ft.acted_last[n])
            return float(put[folder] if folder != seat_a else -put[folder])
        c = float(min(put))
        sa, so = strength(hole[seat_a], b), strength(hole[1 - seat_a], b)
        return c if sa > so else (-c if sa < so else 0.0)

    vals = []
    for seat_a in (0, 1):
        tot, n = 0.0, 0
        for c0 in range(n_cards):
            for c1 in range(n_cards):
                for b in range(n_cards):
                    if len({c0, c1, b}) == 3:
                        tot += walk(0, seat_a, (c0, c1), b)
                        n += 1
        vals.append(tot / n * game.EV_NORMALIZER)
    return np.array([vals[0], vals[1], 0.5 * (vals[0] + vals[1])])
