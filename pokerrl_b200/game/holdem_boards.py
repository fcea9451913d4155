"""Board tables for two-hole-card games: enumeration, suit isomorphism, suit-permutation hand tables (host, integer).

The reference enumerates chance children by recursion over single cards (`PublicTree._make_boards`,
PublicTree.py:193-203), which is wrong for multi-card deals and explodes for Hold'em (SURVEY.md headline 2).  Here a
k-card deal is the set of k-card combinations in lexicographic order - the counts are the reference's own
`DICT_LUT_N_BOARDS` (look_up_table.py:55-60: C(52,5) = 2 598 960 boards for Flop5Holdem) - optionally reduced to one
representative per suit-isomorphism class (134 459 classes) with its orbit size.

Isomorphism contract (DESIGN.md §6): for a suit permutation s, values on board s(b) are the values on b with hands
permuted by s.  A chance parent therefore only needs  W = sum_b (orbit_b / 24) * ev_b  over the representatives and then
ev_parent[h] = sum over the 24 suit permutations s of W[s(h)].
"""
from itertools import combinations, permutations
from math import comb

import numpy as np


def suit_permutation_hand_tables(n_ranks=13, n_suits=4):
    """int16 [n_suits!, R]: table[s][h] = range index of hand h after applying suit permutation s to both cards."""
    n_cards = n_ranks * n_suits
    c1, c2 = np.triu_indices(n_cards, k=1)
    h2i = np.full((n_cards, n_cards), -1, np.int64)
    h2i[c1, c2] = np.arange(c1.size)
    out = []
    for sp in permutations(range(n_suits)):
        sp = np.array(sp)
        m1 = (c1 // n_suits) * n_suits + sp[c1 % n_suits]
        m2 = (c2 // n_suits) * n_suits + sp[c2 % n_suits]
        out.append(h2i[np.minimum(m1, m2), np.maximum(m1, m2)])
    return np.array(out, dtype=np.int16)


def all_boards(cards, k):
    """every k-card combination of `cards` (ascending), lexicographic: int8 [C(len(cards), k), k]"""
    cards = sorted(int(c) for c in cards)
    n = comb(len(cards), k)
    if n > 5_000_000:
        raise ValueError("too many boards to enumerate on the host")
    return np.array(list(combinations(cards, k)), dtype=np.int8).reshape(n, k)


def _combos_52_5():
    """all C(52,5) boards in lexicographic order, built block-wise (first two cards fixed) without 2.6 M Python tuples"""
    a = np.arange(52, dtype=np.int8)
    tri = {}  # 3-combinations of range(m), cached per m
    rows = []
    for c0 in range(52):
        for c1 in range(c0 + 1, 52):
            rest = a[c1 + 1:]
            m = rest.size
            if m < 3:
                continue
            if m not in tri:
                tri[m] = np.array(list(combinations(range(m), 3)), dtype=np.int16)
            t = tri[m]
            blk = np.empty((t.shape[0], 5), np.int8)
            blk[:, 0], blk[:, 1] = c0, c1
            blk[:, 2:] = rest[t]
            rows.append(blk)
    return np.concatenate(rows, axis=0)


def canonical_boards(boards, n_suits=4):
    """Suit-isomorphism classes of a board set that is closed under suit permutations.
    Returns (representatives int8 [n_classes, k] sorted lexicographically, orbit sizes int32 [n_classes])."""
    boards = np.asarray(boards, dtype=np.int64)
    k = boards.shape[1]
    rank, suit = boards // n_suits, boards % n_suits
    best = None
    for sp in permutations(range(n_suits)):
        m = np.sort(rank * n_suits + np.array(sp)[suit], axis=1)
        key = np.zeros(m.shape[0], np.int64)
        for i in range(k):
            key = key * 64 + m[:, i]
        best = key if best is None else np.minimum(best, key)
    uniq, counts = np.unique(best, return_counts=True)
    reps = np.zeros((uniq.size, k), np.int8)
    x = uniq.copy()
    for i in range(k - 1, -1, -1):
        reps[:, i] = x % 64
        x //= 64
    return reps, counts.astype(np.int32)


class BoardSpec:
    """Boards dealt at the (single) chance layer of a two-card game + their weights."""

    def __init__(self, boards, board_prob, board_mult, sym_perm=None, note=""):
        self.boards = np.ascontiguousarray(boards, dtype=np.int8)
        self.board_prob = np.ascontiguousarray(board_prob, dtype=np.float32)
        self.board_mult = np.ascontiguousarray(board_mult, dtype=np.float32)
        self.sym_perm = sym_perm
        self.note = note

    _cache = {}

    @staticmethod
    def full_game(rules, isomorphic=True, deck_subset=None):
        key = (rules.STRING, isomorphic, None if deck_subset is None else tuple(deck_subset))
        if key not in BoardSpec._cache:
            BoardSpec._cache[key] = BoardSpec._full_game(rules, isomorphic, deck_subset)
        return BoardSpec._cache[key]

    @staticmethod
    def _full_game(rules, isomorphic=True, deck_subset=None):
        """All boards of the game's single deal (Flop5Holdem: five cards), as isomorphism classes by default.
        deck_subset: restrict the BOARD cards to these card ids (must be closed under suit permutations when
        isomorphic); hands still range over the whole deck.  The deal probability stays the full-game constant
        1 / C(n_deck - 4, k) unless a subset is given, in which case boards are uniform over the enumerated set."""
        k = rules.N_FLOP_CARDS
        n_deck = rules.N_CARDS_IN_DECK
        if deck_subset is None and isomorphic and n_deck == 52 and k == 5 and rules.N_SUITS == 4:
            # the 134 459 classes of the 2 598 960 five-card boards, precomputed by the code below (data/ file written by
            # tools/gen_iso_classes.py; 8 s of host enumeration otherwise) - counts re-checked on load
            import os
            f = os.path.join(os.path.dirname(os.path.abspath(__file__)), "data", "flop5_iso_classes.npz")
            if os.path.exists(f):
                z = np.load(f)
                reps, orbit = z["boards"], z["orbit"].astype(np.int64)
                if reps.shape == (134459, 5) and int(orbit.sum()) == comb(52, 5):
                    perms = suit_permutation_hand_tables(rules.N_RANKS, rules.N_SUITS)
                    prob = 1.0 / comb(n_deck - 2 * rules.N_HOLE_CARDS, k)
                    return BoardSpec(reps, np.full(reps.shape[0], prob), orbit / float(perms.shape[0]), perms,
                                     "%d suit-isomorphism classes of %d boards" % (reps.shape[0], comb(52, 5)))
        if deck_subset is None:
            boards = _combos_52_5() if (n_deck == 52 and k == 5) else all_boards(range(n_deck), k)
            prob = 1.0 / comb(n_deck - 2 * rules.N_HOLE_CARDS, k)
        else:
            boards = all_boards(deck_subset, k)
            prob = 1.0 / boards.shape[0]
        if not isomorphic:
            return BoardSpec(boards, np.full(boards.shape[0], prob), np.ones(boards.shape[0]), None,
                             "%d boards, no isomorphism" % boards.shape[0])
        reps, orbit = canonical_boards(boards, rules.N_SUITS)
        perms = suit_permutation_hand_tables(rules.N_RANKS, rules.N_SUITS)
        return BoardSpec(reps, np.full(reps.shape[0], prob), orbit / float(perms.shape[0]), perms,
                         "%d suit-isomorphism classes of %d boards" % (reps.shape[0], boards.shape[0]))


class MultiStreetBoards:
    """Boards of a sub-game rooted at a fixed public board with one chance layer per remaining street (e.g. a Hold'em
    flop: layer 1 = turn cards, layer 2 = river cards).  boards[c] = int8 [nb_c, n_cards_out] (children of one parent
    contiguous, ascending card order like PublicTree.py:193-203), parents[c] = int32 [nb_c], prob[c] / mult[c] per
    board.  Deal probability of a k-card deal with m cards already out: 1 / C(n_deck - m - 2 * n_hole, k) - the
    generalisation of the reference's 1 / (N_CARDS_IN_DECK - 2) (StrategyFiller.py:159-166, SURVEY.md appendix A)."""

    def __init__(self, boards, parents, prob, mult, note=""):
        self.boards, self.parents, self.prob, self.mult, self.note = boards, parents, prob, mult, note
        self.n_layers = len(boards) - 1
        self.sym_perm = None

    @staticmethod
    def subgame(rules, root_board, n_layers, root_round, cards_per_layer=None):
        """every card not on the board at each of the next n_layers deals (cards_per_layer: optional restriction of the
        candidate cards of each layer, for small test trees; probabilities stay the full-game constants)"""
        n_deck, n_hole = rules.N_CARDS_IN_DECK, rules.N_HOLE_CARDS
        boards = [np.array([sorted(root_board)], dtype=np.int8).reshape(1, len(root_board))]
        parents, prob, mult = [np.zeros(1, np.int32)], [np.ones(1)], [np.ones(1)]
        rnd = root_round
        for layer in range(1, n_layers + 1):
            rnd += 1
            k = rules.n_cards_dealt_in_transition_to(rnd)
            prev = boards[-1]
            rows, par = [], []
            allowed = None if cards_per_layer is None else set(cards_per_layer[layer - 1])
            for j in range(prev.shape[0]):
                used = set(prev[j].tolist())
                free = [x for x in range(n_deck) if x not in used and (allowed is None or x in allowed)]
                for combo in combinations(free, k):
                    rows.append(list(prev[j]) + list(combo))
                    par.append(j)
            boards.append(np.array(rows, dtype=np.int8).reshape(len(rows), prev.shape[1] + k))
            parents.append(np.array(par, dtype=np.int32))
            prob.append(np.full(len(rows), 1.0 / comb(n_deck - prev.shape[1] - 2 * n_hole, k)))
            mult.append(np.ones(len(rows)))
        return MultiStreetBoards(boards, parents, prob, mult,
                                 "sub-game at board %s, %s boards per layer" % (list(root_board), [b.shape[0] for b in boards]))


def board_class_map(spec):
    """Deal map of a full-game, suit-isomorphic `BoardSpec` of a 52-card, 5-board-card game: for each of the C(52,5) boards,
    indexed by the lexicographic rank of the sorted board (the order of `_combos_52_5`), the class it belongs to (int32, row
    of `spec.boards`) and the suit permutation s (uint8, row of `spec.sym_perm`) that maps the board onto that class's
    representative.  A hand h dealt on the board plays as hand `spec.sym_perm[s][h]` on the representative."""
    reps, sp = np.asarray(spec.boards), spec.sym_perm
    if sp is None or reps.shape != (134459, 5):
        raise ValueError("a board -> class map needs the full game's suit-isomorphism classes (BoardSpec.full_game); a spec over "
                         "a deck subset or without isomorphism has no strategy for most dealt boards")
    if getattr(spec, "_class_map", None) is None:
        boards = _combos_52_5().astype(np.int64)
        rank, suit = boards // 4, boards % 4
        rkey = np.zeros(reps.shape[0], np.int64)
        for i in range(5):
            rkey = rkey * 64 + reps[:, i].astype(np.int64)
        cls = np.full(boards.shape[0], -1, np.int32)
        perm = np.zeros(boards.shape[0], np.uint8)
        for s, p in enumerate(permutations(range(4))):  # the row order of suit_permutation_hand_tables
            m = np.sort(rank * 4 + np.array(p)[suit], axis=1)
            k = np.zeros(m.shape[0], np.int64)
            for i in range(5):
                k = k * 64 + m[:, i]
            pos = np.minimum(np.searchsorted(rkey, k), rkey.size - 1)
            hit = (rkey[pos] == k) & (cls < 0)
            cls[hit] = pos[hit]
            perm[hit] = s
        assert (cls >= 0).all()
        spec._class_map = (cls, perm)
    return spec._class_map
