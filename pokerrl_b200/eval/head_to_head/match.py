"""Head-to-head matches between two eval agents and the exact value of such a match.

`play_match(agent_a, agent_b, n_hands, stack_size)` plays `n_hands` hands with agent A in seat 0, then `n_hands` with A in
seat 1 (the layout of LocalHead2HeadMaster._run_eval, PokerRL/eval/head_to_head/LocalHead2HeadMaster.py:81-126), and
returns A's mean winnings in the game's EV unit with the half width of their 95 % confidence interval
(EvaluatorMasterBase._get_95confidence).

  * Device path, when both agents expose `device_policy()` (tabular agents): every hand is one table of the batched env and
    all tables play in lockstep (csrc/h2h.cu).  Hand g is dealt from the env's shuffle stream g and decision k of hand g
    draws its uniform from a counter hash of (seed, g, k), so the result does not depend on `batch_size`; A's chip results
    are summed in int64, so the sums are bit-identical for any batch split.
  * Host path, for any `EvalAgentBase`: the reference's per-hand loop over the agents' own single-table views.  It deals the
    device path's decks of the same seed and hands its uniforms to agents that sample through `EvalAgentBase._uniform`, so
    a seed means the same hands on both paths.

`exact_head_to_head(agent_a, agent_b, stack_size)` is the expected value of the same match, from one value pass over the
public tree with seat-0 rows of one agent's table and seat-1 rows of the other's.
"""
import ctypes as C
import math

import numpy as np
import torch

from pokerrl_b200 import _native as nat
from pokerrl_b200.game.batched_env import env_config


def _confidence(s, q, n, ev_normalizer):
    """mean and 95 % half width (population std, like numpy's std) from integer sums of chips and squared chips"""
    var = (q * n - s * s) / float(n * n)
    return s / float(n) * ev_normalizer, 1.96 * math.sqrt(max(var, 0.0)) / math.sqrt(n) * ev_normalizer


def counter_uniforms(seed, hands, max_decisions):
    """float64 [len(hands), max_decisions]: the uniforms the device path draws for decisions 0.. of the given global hands
    (the counter hash of csrc/h2h.cu), for replaying device hands through the host loop"""
    m = np.uint64(0xFFFFFFFFFFFFFFFF)

    def mix(z):
        z = (z + np.uint64(0x9E3779B97F4A7C15)) & m
        z = ((z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)) & m
        z = ((z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)) & m
        return z ^ (z >> np.uint64(31))

    with np.errstate(over="ignore"):
        g = np.asarray(hands, np.uint64)[:, None]
        k = np.arange(max_decisions, dtype=np.uint64)[None, :]
        x = mix(mix(np.uint64(seed) ^ mix(g)) + k)
    return (x >> np.uint64(11)).astype(np.float64) * 2.0 ** -53


def deal(env_bldr, stack_size, seed, hand0, n, device=None):
    """int8 [n, n_deck]: the decks of global hands hand0 .. hand0 + n of the device path"""
    dev = torch.device(device if device is not None else "cuda")
    cfg = env_config(env_bldr.env_cls, env_bldr.args_for_stack(stack_size), n)
    state = torch.zeros((nat.lib().prl_env_state_fields(), n), dtype=torch.int32, device=dev)
    deck = torch.zeros((n, cfg.n_deck), dtype=torch.int8, device=dev)
    with torch.cuda.device(dev):
        nat.call("prl_env_reset", C.byref(cfg), C.c_void_p(state.data_ptr()), C.c_void_p(deck.data_ptr()), None, None,
                 int(seed), int(hand0), 1, _stream(dev))
    return deck.cpu().numpy()


def _stream(dev):
    return C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def play_match(agent_a, agent_b, n_hands, stack_size, seed=0, batch_size=1 << 20, device=None):
    """(mean, half width of the 95 % interval) of agent A's winnings per hand over n_hands hands per seat"""
    d = play_match_details(agent_a, agent_b, n_hands, stack_size, seed=seed, batch_size=batch_size, device=device)
    return d["mean"], d["half_width"]


def play_match_details(agent_a, agent_b, n_hands, stack_size, seed=0, batch_size=1 << 20, device=None, decks=None,
                       uniforms=None, winnings=False, host_loop=False):
    """play_match with everything it computed: dict(mean, half_width, sum, sum_sq (int chips), n, desync, path, winnings =
    float32 [2 n_hands] per hand if asked).  decks: int8 [2 n_hands, n_deck] and uniforms: float64 [2 n_hands, k] replace the
    deals and the decision uniforms (replays); host_loop forces the per-hand loop."""
    for e in (agent_a, agent_b):
        e.set_stack_size(stack_size)
    get_pol = lambda e: getattr(e, "device_policy", None)  # noqa: E731
    if not host_loop and get_pol(agent_a) is not None and get_pol(agent_b) is not None:
        return _play_device(agent_a, agent_b, n_hands, stack_size, seed, batch_size, device, decks, uniforms, winnings)
    return _play_host(agent_a, agent_b, n_hands, stack_size, decks, uniforms, seed)


def _play_device(agent_a, agent_b, n_hands, stack_size, seed, batch_size, device, decks, uniforms, want_winnings):
    pa, pb = agent_a.device_policy(device), agent_b.device_policy(device)
    if pa["fingerprint"] != pb["fingerprint"]:
        raise ValueError("the two agents' tables belong to different public trees (stack / bet set)")
    dev = pa["table"].device
    bldr = agent_a.env_bldr
    game, args = bldr.env_cls, bldr.args_for_stack(stack_size)
    total = 2 * int(n_hands)
    sums = torch.zeros(2, dtype=torch.int64, device=dev)
    desync = torch.zeros(1, dtype=torch.int64, device=dev)
    out = torch.empty(total, dtype=torch.float32, device=dev) if want_winnings else None
    max_dec = 0 if uniforms is None else int(np.asarray(uniforms).shape[1])
    ptr = lambda t: None if t is None else C.c_void_p(t.data_ptr())  # noqa: E731
    nf = nat.lib().prl_env_state_fields()
    with torch.cuda.device(dev):
        st = _stream(dev)
        for h0 in range(0, total, int(batch_size)):
            nb = min(int(batch_size), total - h0)
            cfg = env_config(game, args, nb)
            state = torch.zeros((nf, nb), dtype=torch.int32, device=dev)
            deck = torch.zeros((nb, cfg.n_deck), dtype=torch.int8, device=dev)
            rew = torch.zeros((nb, 2), dtype=torch.float64, device=dev)
            actions = torch.empty(nb, dtype=torch.int32, device=dev)
            node, n_dec, chips = (torch.empty(nb, dtype=torch.int32, device=dev) for _ in range(3))
            perm = torch.empty(nb, dtype=torch.uint8, device=dev)
            if decks is not None:
                deck.copy_(torch.as_tensor(np.asarray(decks[h0:h0 + nb]), dtype=torch.int8))
            u = None
            if uniforms is not None:
                u = torch.as_tensor(np.ascontiguousarray(uniforms[h0:h0 + nb], np.float64)).to(dev)
            h = nat.PrlH2H(n_envs=nb, n_range=pa["n_range"], n_hole=pa["n_hole"], chance_by_class=int(pa["board_class"] is not None),
                           max_decisions=max_dec, seat_swap_at=int(n_hands), hand0=h0, seed=int(seed))
            for f in ("kind", "first_child", "n_children", "first_slot", "action", "board_class", "board_perm", "sym_perm"):
                setattr(h, f, ptr(pa[f]))
            h.table_a, h.table_b, h.ld_a, h.ld_b = ptr(pa["table"]), ptr(pb["table"]), pa["ld"], pb["ld"]
            h.uniforms, h.node, h.n_dec, h.perm, h.chips, h.desync = ptr(u), ptr(node), ptr(n_dec), ptr(perm), ptr(chips), ptr(desync)
            nat.call("prl_env_reset", C.byref(cfg), ptr(state), ptr(deck), None, None, int(seed), h0, int(decks is None), st)
            nat.call("prl_h2h_init", C.byref(h), ptr(actions), st)
            for step in range(pa["n_levels"]):
                nat.call("prl_h2h_step", C.byref(h), C.byref(cfg), ptr(state), ptr(deck), ptr(rew), ptr(actions), st)
                nat.call("prl_env_step", C.byref(cfg), ptr(state), ptr(deck), ptr(actions), None, ptr(rew), None, None,
                         int(seed), step, 0, st)
            nat.call("prl_h2h_step", C.byref(h), C.byref(cfg), ptr(state), ptr(deck), ptr(rew), ptr(actions), st)
            nat.call("prl_h2h_collect", C.byref(h), float(cfg.reward_scalar), float(game.EV_NORMALIZER), ptr(sums),
                     None if out is None else ptr(out[h0:h0 + nb]), st)
    n_bad = int(desync.item())
    if n_bad:
        raise RuntimeError("head-to-head: %d tables left the agents' public tree (acting seat or terminal state disagreed with "
                           "the env)" % n_bad)
    s, q = (int(x) for x in sums.cpu().tolist())
    mean, half = _confidence(s, q, total, game.EV_NORMALIZER)
    return {"mean": mean, "half_width": half, "sum": s, "sum_sq": q, "n": total, "desync": n_bad, "path": "device",
            "winnings": None if out is None else out.cpu().numpy()}


_MAX_HOST_DECISIONS = 256  # uniforms drawn per hand on the host path (a hand takes at most "tree depth" decisions)


def _play_host(agent_a, agent_b, n_hands, stack_size, decks, uniforms, seed):
    """LocalHead2HeadMaster._run_eval (:81-126) on single-table views of the device engine"""
    from pokerrl_b200.eval._.EvaluatorMasterBase import EvaluatorMasterBase
    bldr = agent_a.env_bldr
    env = bldr.get_new_env(is_evaluating=True, stack_size=stack_size)
    lut, nh = bldr.lut_holder, bldr.rules.N_HOLE_CARDS
    agents = [agent_a, agent_b]
    winnings = np.empty(2 * n_hands, dtype=np.float32)
    draws = []
    for e in agents:
        e._uniform = lambda: draws.pop(0)  # both agents draw from the hand's stream, in decision order
    try:
        for seat_a in range(2):
            for i in range(n_hands):
                g = seat_a * n_hands + i
                csd = None
                if decks is not None:
                    d = np.asarray(decks[g])
                    csd = {"hand": [lut.get_2d_cards(d[p * nh:(p + 1) * nh]) for p in range(2)],
                           "deck": {"deck_remaining": lut.get_2d_cards(d[2 * nh:])}}
                if decks is None:
                    d = deal(bldr, stack_size, seed, g, 1)[0]
                    csd = {"hand": [lut.get_2d_cards(d[p * nh:(p + 1) * nh]) for p in range(2)],
                           "deck": {"deck_remaining": lut.get_2d_cards(d[2 * nh:])}}
                u = uniforms[g] if uniforms is not None else counter_uniforms(seed, [g], _MAX_HOST_DECISIONS)[0]
                draws[:] = [float(x) for x in u]
                _, r, done, _ = env.reset(deck_state_dict=csd)
                for e in agents:
                    e.reset(deck_state_dict=env.cards_state_dict())
                while not done:
                    p = env.current_player.seat_id
                    me, other = (agents[0], agents[1]) if p == seat_a else (agents[1], agents[0])
                    a, _ = me.get_action(step_env=True, need_probs=False)
                    other.notify_of_action(p_id_acted=p, action_he_did=a)
                    _, r, done, _ = env.step(a)
                winnings[g] = r[seat_a] * env.REWARD_SCALAR * env.EV_NORMALIZER
    finally:
        for e in agents:
            e.__dict__.pop("_uniform", None)
    mean, half = EvaluatorMasterBase._get_95confidence(winnings)
    return {"mean": mean, "half_width": half, "n": 2 * n_hands, "desync": 0, "path": "host", "winnings": winnings}


def exact_head_to_head(agent_a, agent_b, stack_size):
    """Expected winnings of agent A per hand (game EV unit), averaged over A's two seats: one reach + value pass over the
    public tree with seat-0 rows of one agent's table and seat-1 rows of the other's, then sum_h reach_root[p, h] *
    ev[p, root, h] for A's seat p.  Needs tabular agents on the same tree; trees the level engine builds (the Leduc family,
    Flop5Holdem push / fold).  Full-game Flop5Holdem would need on the order of 100 GB on the level engine."""
    from pokerrl_b200.game.PublicTree import PublicTree
    for e in (agent_a, agent_b):
        e.set_stack_size(stack_size)
    ft, fp = agent_a.own_tree()
    if agent_b.own_tree()[1] != fp:
        raise ValueError("the two agents' tables belong to different public trees (stack / bet set)")
    if ft.rules.N_HOLE_CARDS == 2 and bool((ft.kind == 2).any()):
        raise NotImplementedError("exact head-to-head values of two-card trees with a deal need the level engine's full-game "
                                  "tree (~100 GB for Flop5Holdem); use play_match")
    R = ft.R
    rows = [np.asarray(e._rows(0, ft.n_slots), np.float32) for e in (agent_a, agent_b)]
    slot_seat = ft.kind[ft.parent[np.nonzero(ft.slot >= 0)[0]]]  # seat acting at the parent of each slot (flat == slot order)
    ev_norm = agent_a.env_bldr.env_cls.EV_NORMALIZER
    vals = []
    for seat_a in range(2):
        at = np.where((slot_seat == seat_a)[:, None], rows[0], rows[1])
        tree = PublicTree(env_bldr=agent_a.env_bldr, stack_size=stack_size, stop_at_street=None)
        tree.build_tree()
        tree.set_strategy_table(at)
        tree.compute_ev()
        reach, ev = tree._host("reach"), tree._host("ev")
        vals.append(float(np.sum(reach[seat_a, 0, :R].astype(np.float64) * ev[seat_a, 0, :R].astype(np.float64))) * ev_norm)
    return 0.5 * (vals[0] + vals[1])
