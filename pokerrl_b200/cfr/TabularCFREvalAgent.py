"""Tabular CFR `EvalAgent` (SURVEY.md §8f N1): a concrete `EvalAgentBase` backed by the average-strategy table of a
`pokerrl_b200.cfr` solver, so that the solver's result can be handed to the evaluators (`LocalBRMaster`) and stored /
restored (`store_to_disk` / `load_from_disk`).  The reference ships no concrete tabular agent (EvalAgentBase.py is
abstract); the query contract is `StrategyFiller._fill_with_agent_policy` (StrategyFiller.py:88-116).

The agent also plays at its own table (`reset` / `get_action` / `notify_of_action`, EvalAgentBase.py:52-63, 128-158): it
tracks the node of its public tree the table has reached - by action, and at a deal by the board (one-card games: the rank
of the dealt card among the cards not on the board; Flop5Holdem: the board's suit-isomorphism class, with the suit
permutation that maps the board onto the class's representative) - and answers for that node whenever no public-tree node
was set.  Head-to-head matches and LBR play against it this way."""
import numpy as np

from pokerrl_b200 import _native as nat
from pokerrl_b200.rl.base_cls.EvalAgentBase import EvalAgentBase


def tree_fingerprint(ft):
    """structural identity of a flat tree: slot count + hash of kinds / fan-outs / actions / pots"""
    import hashlib
    h = hashlib.sha1()
    for a in (ft.kind, ft.n_children, ft.action, ft.pot):
        h.update(np.ascontiguousarray(a).tobytes())
    return (int(ft.n_slots), h.hexdigest())


def average_strategy_table(solver):
    """float32 [n_slots, R] average strategy of a CFRSolver (host copy), normalised like the reference's `avg_strat`."""
    ft, R = solver.ft, solver.ft.R
    if solver.algo == nat.ALGO_CFR_PLUS:
        if solver.iter_counter <= solver.delay:
            raise RuntimeError("CFR+ has no average strategy before iteration delay+1")
        src = solver.bufs.strat if solver.iter_counter == solver.delay + 1 else solver.bufs.avg
        return src[:, :R].float().cpu().numpy()
    s = solver.bufs.avg[:, :R].cpu().numpy()
    out = np.empty_like(s)
    for n in np.nonzero((ft.kind <= 1) & (ft.first_child >= 0))[0]:
        a, fs = ft.n_children[n], ft.first_slot[n]
        tot = s[fs:fs + a].sum(axis=0, keepdims=True)
        with np.errstate(divide="ignore", invalid="ignore"):
            out[fs:fs + a] = np.where(tot == 0, np.float32(1.0 / a), s[fs:fs + a] / tot)
    return out


def board_strategy_table(solver, ft):
    """float32 [ft.n_slots, ld] device tensor: the average strategy of a board-engine solver (`BoardCFRSolver`) in the slot
    order of the flat tree `ft` over the solver's boards, normalised like `average_strategy_table` (CFR+ at iteration
    delay + 1: regret matching of the regret rows, since the board engine stores no strategy rows)"""
    import torch
    if solver.algo_name == "CFRPlus" and solver.iter_counter <= solver.delay:
        raise RuntimeError("CFR+ has no average strategy before iteration delay+1")
    regret, avg = solver.natural_tables(ft)
    cfr_plus = solver.algo_name == "CFRPlus"
    if cfr_plus and solver.iter_counter > solver.delay + 1:
        return avg
    tab = regret.clamp_(min=0) if cfr_plus else avg
    del regret, avg
    dev = tab.device
    child = np.nonzero(ft.slot >= 0)[0]  # flat order == slot order
    dec = np.nonzero((ft.kind <= 1) & (ft.first_child >= 0))[0]
    dec_idx = np.full(ft.n_nodes, -1, np.int64)
    dec_idx[dec] = np.arange(dec.size)
    seg = torch.from_numpy(dec_idx[ft.parent[child]]).to(dev)
    inv_a = torch.from_numpy(1.0 / ft.n_children[dec].astype(np.float32)).to(dev)
    tot = torch.zeros((dec.size, tab.shape[1]), dtype=torch.float32, device=dev)
    tot.index_add_(0, seg, tab)
    CH = 1 << 17
    for i in range(0, tab.shape[0], CH):
        sg = seg[i:i + CH]
        t = tot[sg]
        tab[i:i + CH] = torch.where(t == 0, inv_a[sg][:, None].expand_as(t), tab[i:i + CH] / torch.where(t == 0, 1.0, t))
    return tab


class TabularCFREvalAgent(EvalAgentBase):
    EVAL_MODE_AVG = "AVG"
    ALL_MODES = [EVAL_MODE_AVG]

    def __init__(self, t_prof, mode=None, device=None):
        super().__init__(t_prof=t_prof, mode=mode or self.EVAL_MODE_AVG, device=device)
        self._table = None  # float32 [n_slots, R (or ld)]: rows in the flat tree's slot order; numpy, or a torch device tensor
        self._n_actions = self.env_bldr.N_ACTIONS
        self._trees = {}  # stack size -> (FlatTree, fingerprint) of the agent's own table
        self._tnode, self._tperm = 0, 0  # tracked node of the agent's own table and the dealt board's suit permutation
        self._dev_cache = None

    def update_weights(self, weights_for_eval_agent):
        """weights: float32 [n_slots, R] table, or (table, fingerprint) with the structural fingerprint of the tree the table
        belongs to (tree_fingerprint); with a fingerprint, querying the agent on a different tree raises.  A torch CUDA tensor
        (rows may be wider than R) stays on its device without a host copy."""
        fp = None
        if isinstance(weights_for_eval_agent, tuple):
            weights_for_eval_agent, fp = weights_for_eval_agent
        if _is_cuda_tensor(weights_for_eval_agent):
            self._table = weights_for_eval_agent.float().contiguous()
        else:
            self._table = np.ascontiguousarray(weights_for_eval_agent, dtype=np.float32)
        self._fingerprint = fp
        self._dev_cache = None

    @classmethod
    def from_cfr(cls, t_prof, cfr, tree_idx=0):
        """the average strategy of `cfr`'s solver for stack `tree_idx`: level engine (host table) or board engine (full-game
        flat tree, device table)"""
        agent = cls(t_prof=t_prof)
        solver = cfr.solvers[tree_idx]
        if getattr(solver, "ft", None) is not None:
            agent.update_weights((average_strategy_table(solver), tree_fingerprint(solver.ft)))
            return agent
        from pokerrl_b200.game.flat_tree import FlatTree
        ft = FlatTree(solver.game_cls, solver.env_args, board_spec=solver.spec_full)
        agent.update_weights((board_strategy_table(solver, ft), tree_fingerprint(ft)))
        agent._trees[_stack_key(solver.env_args.starting_stack_sizes_list)] = (ft, agent._fingerprint)
        return agent

    def can_compute_mode(self):
        return self._table is not None

    def _rows(self, fs, a, hands=None):
        """float32 [a, R] table rows fs .. fs + a (hands: optional row permutation of the hands)"""
        t = self._table[fs:fs + a]
        if _is_cuda_tensor(t):
            t = t.cpu().numpy()
        t = t[:, :self.env_bldr.rules.RANGE_SIZE]
        return t if hands is None else t[:, hands]

    def get_a_probs_for_each_hand(self):
        """[RANGE_SIZE, N_ACTIONS] with the node's probabilities at its allowed actions, 0 elsewhere: the public-tree node
        set by set_to_public_tree_node_state, else the node the agent's own table has reached"""
        node = self._node
        if node is None:
            return self._probs_at_own_table()
        ft = node.tree.flat
        if getattr(self, "_fingerprint", None) is not None and tree_fingerprint(ft) != self._fingerprint:
            raise ValueError("this agent's table was computed on a different public tree (stack / bet set / slot order): "
                             "build one agent per evaluated tree (TabularCFREvalAgent.from_cfr(..., tree_idx=...))")
        fs, a = ft.first_slot[node.idx], ft.n_children[node.idx]
        out = np.zeros((ft.R, self._n_actions), np.float32)
        out[:, node.allowed_actions] = self._rows(fs, a).T
        return out

    # ---- the agent's own table
    def own_tree(self):
        """(FlatTree, fingerprint) of the public tree at the agent's stack size (built once per stack size)"""
        key = _stack_key(self._stack_size)
        if key not in self._trees:
            from pokerrl_b200.game.flat_tree import FlatTree
            ft = FlatTree(self.env_bldr.env_cls, self.env_bldr.args_for_stack(self._stack_size))
            self._trees[key] = (ft, tree_fingerprint(ft))
        ft, fp = self._trees[key]
        if getattr(self, "_fingerprint", None) is not None and fp != self._fingerprint:
            raise ValueError("this agent's table was computed on a different public tree than the one of stack size %r"
                             % (self._stack_size,))
        return ft, fp

    def _deal_map(self, ft):
        from pokerrl_b200.game.holdem_boards import board_class_map
        return board_class_map(ft.board_spec)

    def _probs_at_own_table(self):
        ft, _ = self.own_tree()
        n = self._tnode
        if ft.kind[n] > 1 or ft.first_child[n] < 0:
            raise RuntimeError("the agent's table is not at a decision node (node %d, kind %d)" % (n, ft.kind[n]))
        fs, a, fc = ft.first_slot[n], ft.n_children[n], ft.first_child[n]
        hands = ft.board_spec.sym_perm[self._tperm].astype(np.int64) if self._needs_deal_map(ft) else None
        out = np.zeros((ft.R, self._n_actions), np.float32)
        out[:, ft.action[fc:fc + a]] = self._rows(fs, a, hands).T
        return out

    @staticmethod
    def _needs_deal_map(ft):
        return ft.rules.N_HOLE_CARDS == 2 and bool((ft.kind == 2).any())

    def _advance(self, action):
        """move the tracked node by `action` (just applied at the agent's table) and through a deal by the dealt board"""
        ft, _ = self.own_tree()
        n = self._tnode
        fc, a = ft.first_child[n], ft.n_children[n]
        kids = ft.action[fc:fc + a] if (ft.kind[n] <= 1 and fc >= 0) else np.zeros(0, np.int32)
        if int(action) not in kids:  # an action the table legalised (e.g. a call where calling first is not allowed):
            from pokerrl_b200.game.poker_env import _F  # follow the fold / call the env applied instead
            last_type = int(self.internal_env._state()[0][_F["last_type"]])
            action = last_type if last_type in (0, 1) else action
        hit = np.nonzero(kids == int(action))[0]
        if len(hit) != 1:
            raise RuntimeError("action %d is not a child of the agent's node %d" % (action, n))
        n = fc + int(hit[0])
        if ft.kind[n] == 2:
            env = self.internal_env
            board = np.asarray(env._state()[1][2 * ft.rules.N_HOLE_CARDS:]).astype(np.int64)
            if self._needs_deal_map(ft):
                cls, perm = self._deal_map(ft)
                b = np.sort(board[:5])
                r = _lex_rank_52_5(b)
                j, self._tperm = int(cls[r]), int(perm[r])
            else:
                rnd = env.current_round
                n_prev = ft.rules.n_cards_out_at(rnd - 1)
                card = int(board[n_prev])
                j = card - int(np.sum(board[:n_prev] < card))
            n = ft.first_child[n] + j
        self._tnode = int(n)

    def reset(self, deck_state_dict=None):
        super().reset(deck_state_dict=deck_state_dict)
        self._node, self._tnode, self._tperm = None, 0, 0

    def get_action(self, step_env=True, need_probs=False):
        action, probs = super().get_action(step_env=step_env, need_probs=need_probs)
        if step_env:
            self._advance(action)
        return action, probs

    def notify_of_action(self, p_id_acted, action_he_did):
        super().notify_of_action(p_id_acted, action_he_did)
        self._advance(action_he_did)

    def notify_of_raise_frac_action(self, p_id_acted, frac):
        fracs = self.internal_env.bet_sizes_list_as_frac_of_pot
        if fracs is None:
            return self.notify_of_action(p_id_acted, 2)
        hit = [i for i, f in enumerate(fracs) if abs(float(f) - float(frac)) <= 1e-9 * max(1.0, abs(float(f)))]
        if not hit:
            raise ValueError("pot fraction %r is not in this table's bet set %r" % (frac, fracs))
        self.notify_of_action(p_id_acted, 2 + hit[0])

    def env_state_dict(self):
        d = dict(super().env_state_dict())
        d["tabular_node"] = (self._tnode, self._tperm)
        return d

    def load_env_state_dict(self, state_dict):
        super().load_env_state_dict(state_dict)
        self._tnode, self._tperm = state_dict["tabular_node"]

    def device_policy(self, device=None):
        """what the head-to-head kernel (csrc/h2h.cu) reads for this agent at its current stack size: the table on the
        device, the flat tree's lookup arrays and, for two-card trees with a deal, the board -> (class, suit permutation)
        map.  Dict of torch tensors + scalars; built once per stack size and device."""
        import torch
        ft, fp = self.own_tree()
        dev = torch.device(device if device is not None else (self._table.device if _is_cuda_tensor(self._table) else "cuda"))
        key = (_stack_key(self._stack_size), str(dev))
        if self._dev_cache is not None and self._dev_cache[0] == key:
            return self._dev_cache[1]
        up = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dt)).to(dev)  # noqa: E731
        tab = self._table.to(dev) if _is_cuda_tensor(self._table) else up(self._table, np.float32)
        pol = {"fingerprint": fp, "table": tab, "ld": int(tab.shape[1]), "n_range": ft.R, "n_hole": ft.rules.N_HOLE_CARDS,
               "n_levels": ft.n_levels, "kind": up(ft.kind, np.int8), "first_child": up(ft.first_child, np.int32),
               "n_children": up(ft.n_children, np.int32), "first_slot": up(ft.first_slot, np.int32),
               "action": up(ft.action, np.int32), "board_class": None, "board_perm": None, "sym_perm": None}
        if self._needs_deal_map(ft):
            cls, perm = self._deal_map(ft)
            pol.update(board_class=up(cls, np.int32), board_perm=up(perm, np.uint8), sym_perm=up(ft.board_spec.sym_perm, np.int16))
        self._dev_cache = (key, pol)
        return pol

    def get_a_probs_for_public_tree(self, tree):
        """all decision nodes at once: [n_decision, R, N_ACTIONS] on the tree's device (one scatter of the table rows)"""
        import torch
        ft = tree.flat
        if getattr(self, "_fingerprint", None) is not None and tree_fingerprint(ft) != self._fingerprint:
            raise ValueError("this agent's table was computed on a different public tree")
        dev = tree.dtree.device
        dec = tree.decision_nodes()
        dec_idx = np.full(ft.n_nodes, -1, np.int64)
        dec_idx[dec] = np.arange(dec.size)
        child = np.nonzero(ft.slot >= 0)[0]
        out = torch.zeros((dec.size, ft.R, self._n_actions), dtype=torch.float32, device=dev)
        tab = self._rows(0, ft.n_slots) if not _is_cuda_tensor(self._table) else self._table[:, :ft.R]
        tab = torch.as_tensor(tab).to(dev)  # [n_slots, R]
        out[torch.from_numpy(dec_idx[ft.parent[child]]).to(dev), :, torch.from_numpy(ft.action[child].astype(np.int64)).to(dev)] = tab
        return out

    def _state_dict(self):
        return {"table": self._table.cpu().numpy() if _is_cuda_tensor(self._table) else self._table, "fingerprint": getattr(self, "_fingerprint", None)}

    def _load_state_dict(self, state):
        self._table = state["table"]
        self._dev_cache = None
        self._fingerprint = state.get("fingerprint")


def _is_cuda_tensor(x):
    import torch
    return isinstance(x, torch.Tensor) and x.is_cuda


def _stack_key(stack_size):
    return None if stack_size is None else tuple(int(s) for s in stack_size)


def _lex_rank_52_5(b):
    """lexicographic rank of a sorted 5-card board among all C(52,5) (the order of holdem_boards._combos_52_5)"""
    from math import comb
    return comb(52, 5) - 1 - sum(comb(51 - int(c), 5 - i) for i, c in enumerate(b))
