/*
 * pokerrl_b200 — C ABI of the B200-native tabular CFR / public-tree / best-response path.
 *
 * Drop-in boundary (SURVEY.md §8b).  The reference has no native code on this path — its only FFI precedent is the
 * ctypes convention of PokerRL/_/CppWrapper.py:10-27 (caller allocates every buffer, native code only writes into
 * them, plain pointers and sizes, no ownership transfer).  This header keeps that convention: every pointer marked
 * DEVICE is a raw CUDA device pointer owned by the caller (a torch tensor's data_ptr()), every call is asynchronous
 * on the given CUDA stream, returns 0 on success or a non-zero code with a message in prl_last_error().
 *
 * Each entry point cites the reference interface it replaces (file:line under PokerRL/).
 *
 * Vector layout: every per-node vector is a row of `ld` floats (ld >= n_range, row h = hand / range index in the
 * reference's LUT order: one-card games h = 1D card id; two-card games h = LUT_HOLE_CARDS_2_IDX[c1,c2]).  Per-node
 * arrays are player-major: reach/ev/ev_br = float[2][n_nodes][ld].  Tables (regret, strategy, average) have one row
 * per child of a decision node ("slot"): float[n_slots][ld].
 */
#ifndef POKERRL_B200_H
#define POKERRL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* prl_stream_t; /* cudaStream_t */

/* bumped whenever a struct below changes; prl_abi_version() returns the value the library was built with
   (2: prl_tree_t gained board_hand_rec / node_rec2 / work_rec2 / level_nfold; 3: board engine, legacy LUT natives;
    4: prl_board_sweep / prl_board_trunk take the algorithm; prl_tree_t gained the all-in terminals of two-card games: level_nallin / allin_nodes / allin_pot / allin_tiles /
    allin_partial) */
#define PRL_ABI_VERSION 4

/* node kinds (game/_/tree/_/nodes.py:8-62 + ValueFiller.py:34-62) */
enum {
    PRL_KIND_P0 = 0,             /* player 0 acts next */
    PRL_KIND_P1 = 1,             /* player 1 acts next */
    PRL_KIND_CHANCE = 2,         /* chance acts next ("Ch") */
    PRL_KIND_FOLD = 3,           /* terminal: acted_last folded */
    PRL_KIND_SHOWDOWN = 4,       /* terminal: showdown with complete board */
    PRL_KIND_SHOWDOWN_ALLIN = 5  /* terminal: all-in showdown before the board is complete */
};

/* algorithms (cfr/VanillaCFR.py, cfr/CFRPlus.py, cfr/LinearCFR.py) */
enum { PRL_ALGO_VANILLA = 0, PRL_ALGO_CFR_PLUS = 1, PRL_ALGO_LINEAR = 2 };

/* where a player's strategy comes from in a reach / value pass, and in which precision the reference computes
 * with it (SURVEY.md appendix C) */
enum {
    PRL_STRAT_F32 = 0,       /* float table `strat`                       (after the player's first update)        */
    PRL_STRAT_UNIFORM64 = 1, /* 1.0/A in double                            (StrategyFiller.py:61-62, before it)     */
    PRL_STRAT_AVG_F64 = 2,   /* double table `avg`                         (CFR+ average under numpy>=2)            */
    PRL_STRAT_AVG_SUM = 3,   /* float table `avg` holding reach-weighted sums, normalised on the fly, double math
                                                                           (LinearCFR.py:64-71, VanillaCFR.py:65-72) */
    PRL_STRAT_AVG_F32 = 4    /* float table `avg` used as is, float math   (CFR+ average under numpy<2)             */
};

/* Depth-sorted public tree in HBM (replaces the object tree of game/_/tree/PublicTree.py:111-293, nodes.py). */
typedef struct {
    int32_t n_nodes, n_levels, n_slots;
    int32_t n_range;    /* RANGE_SIZE */
    int32_t ld;         /* row stride in elements */
    int32_t n_hole;     /* hole cards per hand: 1 (Leduc family) or 2 (Hold'em family) */
    int32_t n_deck;     /* N_CARDS_IN_DECK */
    int32_t n_suits;    /* N_SUITS (card c = rank * n_suits + suit) */
    int32_t pair_bonus; /* one-card games: added to the rank of a hand pairing the board (game_rules.py:68-75) */
    int32_t max_actions;
    const int64_t* level_start;  /* HOST int64[n_levels+1]: nodes of depth d are [level_start[d], level_start[d+1]) */
    const int32_t* parent;       /* DEVICE int32[n_nodes], -1 for the root */
    const int32_t* first_child;  /* DEVICE int32[n_nodes], -1 if none; children are contiguous */
    const int32_t* n_children;   /* DEVICE int32[n_nodes] */
    const int32_t* slot;         /* DEVICE int32[n_nodes]: table row of this node as a child of a decision node, else -1 */
    const int8_t* kind;          /* DEVICE int8[n_nodes] */
    const int8_t* acted_last;    /* DEVICE int8[n_nodes]: seat that acted last (folder at fold terminals) */
    const float* pot;            /* DEVICE float[n_nodes]: main pot (chips) */
    const int32_t* board;        /* DEVICE int32[n_nodes]: one-card games: the board card or -1; two-card games: board id */
    const int32_t* order;        /* DEVICE int32[n_nodes]: per level, the node ids of that level sorted by (kind,
                                    n_children) with terminals last - thread t of a level works on node order[t], so a
                                    warp holds nodes of one kind (no divergence); data layout is unaffected */
    const int64_t* level_nonterm; /* HOST int64[n_levels]: number of non-terminal nodes of each level */
    const void* meta;            /* DEVICE 16-byte record per node, filled by prl_pack_node_meta() from the arrays above:
                                    {first_child, first_slot, pot, kind | acted_last | board | n_children}; the sweeps
                                    read node structure only through it (one 128-bit load per node) */
    /* ---- two-hole-card games only (n_hole == 2); NULL / 0 otherwise ------------------------------------------- */
    const int64_t* level_ndec;   /* HOST int64[n_levels]: decision nodes per level (first in `order`, then chance nodes) */
    const int8_t* hand_cards;    /* DEVICE int8[n_range][2]: LUT_IDX_2_HOLE_CARDS */
    int32_t n_boards;            /* rows of the board tables below; node.board indexes them */
    int32_t max_chance_children; /* largest fan-out of a chance node */
    const uint64_t* board_mask;  /* DEVICE uint64[n_boards]: bit c set iff card c lies on the board */
    const float* board_prob;     /* DEVICE float[n_boards]: factor applied to BOTH reach rows when this board is dealt
                                    (1 / C(deck - 4, k) in the full game; hands holding a board card get 0) */
    const float* board_mult;     /* DEVICE float[n_boards]: weight of this board's values in its parent's sum (1, or
                                    orbit size / n_sym for a suit-isomorphism class representative) */
    const int16_t* board_gs;     /* DEVICE int16[n_boards][n_range]: # live hands strictly weaker (-1: hand blocked)   */
    const int16_t* board_ge;     /* DEVICE int16[n_boards][n_range]: # live hands weaker or equal                      */
    const int16_t* board_pos;    /* DEVICE int16[n_boards][n_range]: position in strength order (prl_board_order_tables) */
    const int16_t* board_row_order; /* DEVICE int16[n_boards][n_deck][n_deck-1]: per card, the live hands holding it in
                                       strength order (-1 padded) */
    const uint8_t* board_row_pos;   /* DEVICE uint8[n_boards][n_range][4]: per hand {# weaker in row c1, # weaker in row
                                       c2, # weaker-or-equal in row c1, in row c2} */
    const uint8_t* board_complete;  /* DEVICE uint8[n_boards]: 1 iff the board shows all N_TOTAL_BOARD_CARDS (tables above valid) */
    int32_t n_sym;               /* hand permutations summed at chance parents (24 suit permutations with isomorphism, else 0/1) */
    const int16_t* sym_perm;     /* DEVICE int16[n_sym][n_range] */
    float eq_const;              /* opponent-hand normaliser C(deck,2)/C(deck-2,2) (ValueFiller.py:19 generalised) */
    const void* board_hand_rec;  /* DEVICE int16[n_boards][n_range][8] or NULL: the showdown tables of one hand packed for a
                                    single 16-byte load: {gs, ge, c1*53 + row_pos[0], c1*53 + row_pos[2],
                                    c2*53 + row_pos[1], c2*53 + row_pos[3], 0, 0} (53 = row stride of the card-row
                                    prefix array in shared memory); NULL: the separate tables above are read */
    const void* node_rec2;       /* DEVICE int32[n_nodes][4] or NULL: {parent, slot, first slot of the parent's children,
                                    kind(parent) | n_children(parent) << 8} - the top-down sweep reads a node's structure
                                    with one 16-byte load; NULL: parent / slot / first_child / n_children / kind are read */
    const void* work_rec2;       /* DEVICE int32[n_nodes][4] or NULL, indexed like `order`: {node, first child, first slot of
                                    the children, kind | n_children << 8} for the bottom-up sweep over decision nodes;
                                    terminal entries: {node, board id, pot as float bits, kind | (acted_last & 0xff) << 8} */
    const int64_t* level_nfold;  /* HOST int64[n_levels] or NULL: fold terminals per level (they come first among the
                                    terminals in `order`); lets fold and showdown rows be launched as separate kernels */
    /* two-card games, all-in showdowns before the board is complete (PRL_KIND_SHOWDOWN_ALLIN; the one-card analogue is
       ValueFiller.py:160-175): they come LAST among the terminals of a level in `order`; their values are the dense product
       of the public board's equity matrix with the opponent's reach row (prl_allin_values, tensor cores); one matrix per
       public board such a terminal occurs on. */
    const int64_t* level_nallin; /* HOST int64[n_levels] or NULL (= no such terminals) */
    const int32_t* allin_nodes;  /* HOST int32[sum of level_nallin]: their node ids, ascending (= by level) */
    const float* allin_pot;      /* HOST float[same]: pot of each */
    const void* const* allin_tiles; /* HOST array [same] of DEVICE pointers: the equity matrix of each node's public board as bf16
                                       operand tiles (prl_allin_equity_finish); nodes on the same board share a pointer */
    float* allin_partial;        /* DEVICE scratch, prl_allin_partial_bytes(n_range) bytes */
} prl_tree_t;

/* Caller-owned work buffers. */
typedef struct {
    float* reach;  /* DEVICE float[2][n_nodes][ld]   node.reach_probs */
    float* ev;     /* DEVICE float[2][n_nodes][ld]   node.ev */
    float* ev_br;  /* DEVICE float[2][n_nodes][ld]   node.ev_br (may be NULL when no pass asks for BR) */
    float* regret; /* DEVICE float[n_slots][ld]      node.data["regret"] */
    float* strat;  /* DEVICE float[n_slots][ld]      node.strategy */
    void* avg;     /* DEVICE float|double[n_slots][ld]  node.data["avg_strat"] (CFR+) / ["avg_strat_sum"] */
    void* workspace;          /* DEVICE scratch for the chance-node reductions of two-card games (else NULL) */
    uint64_t workspace_bytes; /* >= 4 * n_chance_per_level * (ceil(max_chance_children / 128) + 1) * ld * 4 bytes */
} prl_buffers_t;

/* library info */
int prl_abi_version(void);
const char* prl_last_error(void);
/* number of CUDA kernels this library has launched so far in this process */
unsigned long long prl_launch_count(void);

/* Packs the per-node structure arrays of `tree` into out_meta = DEVICE int4[n_nodes] (then set tree->meta = out_meta).
 * Call once after uploading a tree (the analogue of PublicTree.build_tree finishing, PublicTree.py:111-126). */
int prl_pack_node_meta(const prl_tree_t* tree, void* out_meta, prl_stream_t stream);

/* StrategyFiller.update_reach_probs (StrategyFiller.py:118-146) for the seats in player_mask (bit p).
 * Writes reach[p] of every node from the root down; root = 1/n_range (PublicTree.py:122-124).
 * strat_mode[p] selects the strategy source of seat p's decision nodes. */
int prl_reach_pass(const prl_tree_t* tree, const prl_buffers_t* buf, int player_mask, const int* strat_mode,
                   prl_stream_t stream);

/* ValueFiller.compute_cf_values_heads_up (ValueFiller.py:21-101) for the seats in player_mask, bottom-up.
 * with_br != 0 also fills ev_br.  Terminal values follow ValueFiller.py:103-175. */
int prl_value_pass(const prl_tree_t* tree, const prl_buffers_t* buf, int player_mask, int with_br,
                   const int* strat_mode, prl_stream_t stream);

/* Root exploitability (ValueFiller.py:95-101): out_expl = DEVICE float[2], chips. */
int prl_root_exploitability(const prl_tree_t* tree, const prl_buffers_t* buf, float* out_expl, prl_stream_t stream);

/* One CFR half-iteration for seat p, fused (replaces _CFRBase.py:123-128 for one p):
 *   bottom-up:  ev[p] of every node; at p's decision nodes regret update (_CFRBase.py:146-185 with the formula of
 *               algo) and regret matching into `strat` (CFRPlus.py:43-63 / LinearCFR.py:33-51 / VanillaCFR.py:32-52)
 *   top-down:   reach[p] of every node with the new strategy (StrategyFiller.py:118-146) and the average-strategy
 *               update of p's nodes (CFRPlus.py:65-87 / LinearCFR.py:53-76 / VanillaCFR.py:54-77)
 * iter = _iter_counter (0-based); delay = CFR+ averaging delay; avg_f64 = `avg` is double. strat_mode as above
 * (entry of seat p is what the value pass reads; after the call seat p's strategy is PRL_STRAT_F32). */
int prl_cfr_half_iteration(const prl_tree_t* tree, const prl_buffers_t* buf, int algo, int p, int iter, int delay,
                           int avg_f64, const int* strat_mode, prl_stream_t stream);

/* n_iters full CFR iterations (_CFRBase.iteration :122-128 without the logging passes) in ONE persistent cooperative
 * kernel launch: for each iteration, for p in (0, 1): value/regret sweep then reach/average sweep, grid barrier
 * between tree levels.  iter0 = _iter_counter of the first iteration; strat_mode = sources at entry (seat p switches
 * to PRL_STRAT_F32 after its first update, exactly like a sequence of prl_cfr_half_iteration calls). */
int prl_cfr_iterations(const prl_tree_t* tree, const prl_buffers_t* buf, int algo, int iter0, int n_iters, int delay,
                       int avg_f64, const int* strat_mode, prl_stream_t stream);

/* Exploitability evaluation in one persistent launch (_CFRBase._log_curr_strat_expl :198-216 / _evaluate_avg_strats
 * :218-262; eval/br/LocalBRMaster.py:67-80): optional reach pass for both seats (do_reach), value pass with best
 * response for both seats, root exploitability -> out_expl = DEVICE float[2] (chips). */
int prl_evaluate(const prl_tree_t* tree, const prl_buffers_t* buf, const int* strat_mode, int do_reach, float* out_expl,
                 prl_stream_t stream);

/* Profiling aid: if set to a DEVICE uint64 buffer (>= 1 + 4*n_levels*n_iters entries), prl_cfr_iterations records
 * %globaltimer (ns) at entry and after every grid barrier; NULL (default) disables it. */
void prl_debug_set_timeline(void* device_u64_buffer);

/* The two sweeps of prl_cfr_half_iteration separately (which: bit 0 = bottom-up value/regret sweep, bit 1 = top-down
 * reach/average sweep); prl_cfr_half_iteration == which 3.  Used to time the sweeps individually. */
int prl_cfr_sweep(const prl_tree_t* tree, const prl_buffers_t* buf, int algo, int p, int iter, int delay, int avg_f64,
                  const int* strat_mode, int which, prl_stream_t stream);

/* Multi-GPU building blocks (two-card trees sharded by board, DESIGN.md §7).  prl_value_levels runs the bottom-up sweep
 * over levels level_hi..level_lo only; algo >= 0 makes it the update sweep of seat upd_p (else a plain value pass, with
 * best response if with_br).  chance_phase 1 stops before the final stage of the chance reduction, leaving the per-node
 * sums in buf->workspace at float offset 4*n_chance*ceil(max_chance_children/128)*ld, laid out [4][n_chance][ld]
 * (array index = 2*seat + {0: ev, 1: ev_br}) so that the caller can all-reduce them over the ranks (the ONE collective
 * of the path, SURVEY.md §8e); chance_phase 2 runs only that final stage; 0 runs whole levels.
 * prl_reach_update is the top-down half of prl_cfr_half_iteration for seat p. */
int prl_value_levels(const prl_tree_t* tree, const prl_buffers_t* buf, int player_mask, int with_br, int algo, int upd_p,
                     int iter, int delay, const int* strat_mode, int level_hi, int level_lo, int chance_phase,
                     prl_stream_t stream);
int prl_reach_update(const prl_tree_t* tree, const prl_buffers_t* buf, int algo, int p, int iter, int delay,
                     prl_stream_t stream);

/* Top-down reach sweep over tree levels level_lo..level_hi only (StrategyFiller.py:118-146); algo >= 0 adds the
 * average-strategy update of seat upd_p (as in prl_cfr_half_iteration). */
int prl_reach_levels(const prl_tree_t* tree, const prl_buffers_t* buf, int player_mask, int algo, int upd_p, int iter,
                     int delay, const int* strat_mode, int level_lo, int level_hi, prl_stream_t stream);

/* Batched StrategyFiller._fill_with_agent_policy (StrategyFiller.py:88-116): probs = DEVICE float[n_decision][n_range]
 * [n_actions] (the agent's get_a_probs_for_each_hand for every decision node at once, EvalAgentBase.py:39-44), dec_of_slot /
 * action_of_slot = DEVICE int32[n_slots] (decision node index and discrete action of every table row) -> out = DEVICE
 * float[n_slots][ld] strategy table (`strat` of prl_buffers_t). */
int prl_gather_agent_policy(const float* probs, int n_actions, const int32_t* dec_of_slot, const int32_t* action_of_slot,
                            int n_slots, int n_range, int ld, float* out, prl_stream_t stream);

/* Strength-order tables of complete boards for the two-card showdown rows: ranks = DEVICE int32[n_boards][n_range]
 * (prl_hand_rank_boards; -1 = blocked) -> gs / ge / pos = DEVICE int16[n_boards][n_range], row_order = DEVICE
 * int16[n_boards][n_deck][n_deck-1], row_pos = DEVICE uint8[n_boards][n_range][4] (see prl_tree_t). */
int prl_board_order_tables(const int32_t* ranks, int n_boards, int n_range, int n_deck, int16_t* gs, int16_t* ge,
                           int16_t* pos, int16_t* row_order, uint8_t* row_pos, prl_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Board-resident CFR+ engine (csrc/cfr_board.cu) for two-card games with ONE chance layer whose post-deal subtree has
 * the compiled shape (Flop5Holdem, PokerRL/game/games.py:222-254: 15 nodes per board).  Replaces, for the post-deal
 * levels, ValueFiller.compute_cf_values_heads_up (ValueFiller.py:21-158), StrategyFiller._update_reach_probs
 * (StrategyFiller.py:118-146) and the regret / matching / averaging of CFRPlus.py:37-87: one persistent kernel walks
 * (board, seat) units with the subtree in registers / shared memory.  Table rows of a board are stored in the board's
 * strength order over the n_live = C(n_deck - 5, 2) hands that hold no board card (stride ldb); the strategy is not
 * stored (regret matching of the regret rows).  The pre-deal trunk stays with the level sweeps above.
 * ------------------------------------------------------------------------------------------------------------------ */
typedef struct {
    int32_t n_boards;  /* boards resident on this device */
    int32_t n_range;   /* 1326 */
    int32_t ld;        /* stride of natural-order rows (trunk vectors) */
    int32_t n_deck;    /* 52 */
    int32_t n_local;   /* nodes of the post-deal subtree, breadth-first, local 0 = first node after the deal */
    int32_t frac_bits; /* the chance-node sums are accumulated as int64 fixed point with this many fraction bits */
    int32_t grid;      /* CTAs of the persistent kernel; 0 = library default (2 per SM) */
    float eq_const;    /* C(deck,2)/C(deck-2,2) (ValueFiller.py:19 generalised) */
    int8_t kind[16], parent[16], first_child[16], n_children[16], acted_last[16];
    float pot[16];
    int64_t row0[16];  /* table row of local node i (a child of a decision node) on board 0; -1: none */
    int32_t row_m[16]; /* row(i, j) = row0[i] + j * row_m[i] (= fan-out of the parent) */
    const void* tables;      /* DEVICE [n_boards][blob bytes] built by prl_board_build_tables */
    const float* board_prob; /* DEVICE float[n_boards]: deal probability applied to both reach rows */
    const float* board_mult; /* DEVICE float[n_boards]: weight in the parent's sum (orbit size / 24 or 1) */
    float* regret;           /* DEVICE float[n_rows][ldb] */
    float* avg;              /* DEVICE float[n_rows][ldb]  CFR+ average strategy */
    int64_t* w_private;      /* DEVICE int64[grid][2][n_range] scratch */
    int64_t* w_total;        /* DEVICE int64[4][n_range]: fixed-point sums over this device's boards of board_mult * root value,
                                natural hand order.  Update sweep: array 0 = ev of the seat; evaluation sweep of seat p:
                                arrays 2p = ev, 2p + 1 = ev_br */
} prl_board_game_t;

/* out[8] = {n_live, ldb, blob bytes per board, byte offset of the int16 hand ids, byte offset of the card rows,
 *           live cards, padded card-row length, nodes of the compiled shape} */
int prl_board_layout(int32_t* out);
int prl_board_grid(void);                              /* default CTA count on the current device */
int prl_board_shape_ok(const prl_board_game_t* g);     /* 1 iff kind / parent / first_child / n_children match */

/* ranks = DEVICE int32[n_boards][1326] (prl_hand_rank_boards), board_mask = DEVICE uint64[n_boards] -> blob */
int prl_board_build_tables(const int32_t* ranks, const uint64_t* board_mask, const int8_t* hand_cards, int n_boards,
                           void* blob, prl_stream_t stream);

/* One sweep over all boards for seat p.  eval == 0: update of p's post-deal rows by `algo` (PRL_ALGO_*; iteration iter,
 * CFR+ averaging delay `delay`); eval != 0: values and best-response values of p with the strategies of p / the opponent
 * taken from src_own / src_opp (0 = regret matching of `regret`, 1 = rows of `avg` as they are (CFR+ average), 2 = rows of
 * `avg` normalised (the reach-weighted sums of Vanilla / Linear CFR)).  trunk_reach_opp = DEVICE float[ld]: reach row of the
 * opponent at the chance node.  Leaves the fixed-point sums in g->w_total (the arrays it produces are zeroed first).
 * Vanilla / Linear CFR (VanillaCFR.py:54-60, LinearCFR.py:53-59): the average is the sum of strategy x own reach x weight with
 * the reach under the NEW strategy, trunk included - known only after the seat's trunk update.  The contribution of the
 * OPPONENT's last update is therefore added by this sweep (defer_w = its weight, 0 = none pending), which walks those rows
 * anyway; p1_only != 0 does nothing else (flush before the average strategy is evaluated or exported). */
int prl_board_sweep(const prl_board_game_t* g, int p, int eval, int src_own, int src_opp, const float* trunk_reach_opp,
                    int iter, int delay, int algo, float defer_w, int p1_only, prl_stream_t stream);

/* out[a][h] = 2^-frac_bits * sum over the n_sym suit permutations of w_total[a][perm(h)] (n_sym <= 1: no symmetrisation),
 * a < n_arr: the chance node's rows for the trunk sweep (after an all-reduce of w_total across GPUs, if sharded). */
int prl_board_collect(const prl_board_game_t* g, int n_arr, const int16_t* sym_perm, int n_sym, float* out, int ld,
                      prl_stream_t stream);

/* The pre-deal trunk (<= 8 nodes, breadth-first ids = flat-tree ids 0 .. n_nodes - 1; exactly one chance node, a leaf here)
 * for prl_board_trunk: one launch replaces the level sweeps over the trunk - ValueFiller.py:64-125 bottom-up from the
 * chance node's sums, CFRPlus.py:37-87 at seat p's nodes, StrategyFiller.py:118-146 for p's reach rows (update form), or
 * values + best response of both seats and the root exploitability (evaluation form, out_expl = DEVICE float[2]). */
typedef struct {
    int32_t n_nodes, chance_node, n_buf_nodes, ld, n_range;
    int32_t mode[2];        /* PRL_STRAT_* source of each seat's trunk strategy (UNIFORM64, F32 or AVG_F32) */
    float eq_const;
    int8_t kind[8], first_child[8], n_children[8], acted_last[8];
    int32_t first_slot[8];
    float pot[8];
    const int8_t* hand_cards; /* DEVICE int8[n_range][2] */
    float* reach;   /* DEVICE float[2][n_buf_nodes][ld] */
    float* ev;
    float* ev_br;
    float* regret;  /* DEVICE float[n_slots][ld] trunk tables (natural hand order) */
    float* strat;
    float* avg;
} prl_trunk_t;

/* peers != NULL fuses the ONE collective of the path into this launch: peers = DEVICE array of n_peers pointers to every rank's
 * w_total buffer in peer-mapped (symmetric) memory, read over NVLink at element offset peer_offset and summed in rank order
 * into w_scratch (DEVICE int64[4][n_range]); the caller orders this launch after all ranks' sweeps with a cross-rank barrier.
 * peers == NULL: g->w_total already holds the global sums (single GPU, or all-reduced by the caller). */
int prl_board_trunk(const prl_board_game_t* g, const prl_trunk_t* t, int eval, int p, int n_sym, const int16_t* sym_perm, int iter,
                    int delay, float* out_expl, const int64_t* const* peers, int n_peers, int64_t peer_offset, int64_t* w_scratch,
                    int algo, prl_stream_t stream);

/* Strength-ordered rows <-> natural-order rows.  row_src / row_dst = DEVICE int64[rows_per_board][2] {row on board 0,
 * stride per board} in the strength-ordered table and in a natural-order table of stride ld. */
int prl_board_permute(const prl_board_game_t* g, int rows_per_board, const int64_t* row_src, const int64_t* row_dst,
                      float* sorted_tab, float* natural_tab, int ld, int to_natural, prl_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * 7-card Hold'em hand evaluation (replaces lib_hand_eval.so; int32 strength, higher = better, identical encoding incl.
 * the quads-kicker quirk - see oracle/hand_eval_oracle.c).  Cards are 1D ids c = rank*4 + suit.
 * ------------------------------------------------------------------------------------------------------------------ */

/* ---------------------------------------------------------------------------------------------------------------
 * All-in showdowns before the board is complete, two-card games (csrc/allin_dense.cu).  The reference enumerates the
 * missing board cards per terminal (ValueFiller.py:160-175 `_get_call_eq_preflop`, one-card games only); here the public
 * state's EQUITY MATRIX  E[h][h'] = sum over the sym_perm permutations q and the completions b of the board of
 * w_b * sign(rank_b(q(h)) - rank_b(q(h'))) (0 where a hand is blocked or the two hands share a card) is built once, stored
 * as three bf16 split planes in tcgen05 operand tiles, and every all-in terminal costs one column of a tensor-core GEMM
 * (BASELINE.json north_star: "tensor cores used only for the dense 1326x1326 Hold'em showdown equity contraction").
 *   prl_allin_equity_accumulate: ec (DEVICE double[n_range][n_range], zeroed by the caller) += sum_b weight[b] * S_b for a chunk
 *     of boards; ranks DEVICE int32[n_boards][n_range] (prl_hand_rank_boards), weight DEVICE double[n_boards] (deal probability
 *     x weight in the parent's sum).
 *   prl_allin_equity_finish: symmetrises over sym_perm (NULL / n_sym <= 1: none), masks hands sharing a card, splits into
 *     three bf16 planes (24 mantissa bits) and writes the operand tiles (prl_allin_tiles_bytes bytes).
 *   prl_allin_values: for column c < n_cols: y_rows[c][h] (and y2_rows[c][h] if y2_rows and y2_rows[c]) =
 *     scale[c] * sum_h' E[h][h'] * x_rows[c][h'].  x_rows / y_rows / y2_rows / scale are HOST arrays (of DEVICE row pointers);
 *     fp32 operands are split into three bf16 planes on the fly, products accumulate in fp32 in tensor memory.
 */
int64_t prl_allin_tiles_bytes(int n_range);
int64_t prl_allin_partial_bytes(int n_range);
int prl_allin_equity_accumulate(const int32_t* ranks, const double* weight, int n_boards, int n_range, double* ec,
                                prl_stream_t stream);
int prl_allin_equity_finish(const double* ec, int n_range, const int8_t* hand_cards, const int16_t* sym_perm, int n_sym,
                            void* tiles, prl_stream_t stream);
int prl_allin_values(const void* tiles, int n_range, const float* const* x_rows, float* const* y_rows, float* const* y2_rows,
                     const float* scale, int n_cols, float* partial, prl_stream_t stream);

/* HoldemRules.get_hand_rank_all_hands_on_given_boards (game_rules.py:213-217) on device buffers:
 * boards = DEVICE int8[n_boards][5], out = DEVICE int32[n_boards][1326] (-1 where the hand is blocked by the board;
 * hand order = LUT_IDX_2_HOLE_CARDS). */
int prl_hand_rank_boards(const int8_t* boards, int n_boards, int32_t* out, prl_stream_t stream);

/* n independent 7-card hands: cards = DEVICE int8[n][7] -> out = DEVICE int32[n] (game_rules.py:219-223 batched). */
int prl_hand_rank_7(const int8_t* cards, int n, int32_t* out, prl_stream_t stream);

/* Local Best Response roll-out (eval/lbr/LocalLBRWorker.py:377-512, _LBRRolloutManager.get_lbr_checkdown_equity): for each of
 * n_queries (LBR hand, dealt board cards, agent range) the probability-weighted check-down equity over EVERY completion of
 * the board.  lbr_hands = DEVICE int8[n][2] (1D cards), boards = DEVICE int8[n][5] (the n_dealt dealt cards first; all
 * queries of a call are on the same street), ranges = DEVICE float[n][1326] (normalised, zero on hands holding an LBR or
 * board card), workspace = DEVICE double[prl_lbr_workspace_doubles(n, n_dealt)], out = DEVICE float[n].
 * first_board_ranks != 0 reproduces a defect of the reference - its board counter `_i` is never advanced
 * (LocalLBRWorker.py:468-512), so every completion is compared on the ranks of the FIRST completion - and exists for
 * parity checks against outputs of the reference; 0 (the product's default) ranks every completion on its own cards. */
long long prl_lbr_workspace_doubles(int n_queries, int n_dealt);
int prl_lbr_checkdown_equity(const int8_t* lbr_hands, const int8_t* boards, int n_dealt, const float* ranges, int n_queries,
                             int first_board_ranks, double* workspace, float* out, prl_stream_t stream);

/* Legacy entry points with the exact native signatures the reference binds through ctypes (HOST arrays of row
 * pointers, PokerRL/_/CppWrapper.py:24-27): CppHandeval.py:22-33 and CppLUT.py:22-35 can load this library unchanged.
 * They stage through device memory and run the kernels above (synchronous). */
int32_t get_hand_rank_52_holdem(int8_t** hand_2d /*[2][2]*/, int8_t** board_2d /*[5][2]*/);
void get_hand_rank_all_hands_on_given_boards_52_holdem(int32_t** out /*[n][1326]*/, int8_t** boards_1d /*[n][5]*/,
                                                       int32_t n, int8_t** idx2holecards, int8_t** card1d_to_2d);
void get_hole_card_2_idx_lut(int16_t** lut /*[52][52]*/);
void get_idx_2_hole_card_lut(int8_t** lut /*[1326][2]*/);
/* bound by CppLibHoldemLuts.__init__ (CppLUT.py:28-35), never called by the reference; its own binary faults on them
 * (INTEGRATION.md §2).  Defined, in-bounds results for the buffer shapes of CppLUT.py:47-72. */
void get_idx_2_flop_lut(int8_t** lut /*[22100][3]: 3-card combinations, lexicographic*/);
void get_idx_2_turn_lut(int8_t** lut /*[52][4]: row i column 0 = card i*/);
void get_idx_2_river_lut(int8_t** lut /*[52][5]: row i column 0 = card i*/);
int8_t get_1d_card(const int8_t* card_2d);
void get_2d_card(int8_t card_1d, int8_t* out_card_2d);

/* ------------------------------------------------------------------------------------------------------------------
 * Batched heads-up PokerEnv (replaces the scalar Python engine PokerRL/game/_/rl_env/base/PokerEnv.py for B tables at
 * once; SURVEY.md §8a row J / appendix B).  One table per thread, integer chips, the reference's action decoding,
 * legalisation, round logic, payouts, rewards and observation layout.
 * ------------------------------------------------------------------------------------------------------------------ */
#define PRL_ENV_MAX_ACTIONS 34

typedef struct {
    int32_t n_envs;
    int32_t kind;          /* 0 = limit-type action space {fold, call, raise} (LimitPokerEnv.py), 1 = discretized pot
                              fractions (DiscretizedPokerEnv.py) */
    int32_t n_actions;     /* env_args.N_ACTIONS */
    int32_t n_rounds;      /* len(ALL_ROUNDS_LIST) */
    int32_t n_round_slots; /* ALL_ROUNDS_LIST[-1] + 1 (one-hot width in the observation) */
    int32_t n_hole, n_ranks, n_suits, n_deck;
    int32_t n_flop, n_turn, n_river;
    int32_t small_blind, big_blind, ante, small_bet, big_bet, round_big_bet_starts;
    int32_t max_raises[4]; /* MAX_N_RAISES_PER_ROUND */
    int32_t first_action_no_call, limit_raise_is_pot, btn_first_postflop, suits_matter;
    int32_t pair_bonus;    /* one-card games: hand strength bonus for pairing the board */
    int32_t start_stack[2];
    int32_t obs_size;      /* 7 + 3 + 2 + 2 + n_round_slots + 6 + n_board_cards * (n_ranks + n_suits) */
    double fracs[32];      /* sorted bet sizes as fractions of the pot (kind 1) */
    double reward_scalar;  /* REWARD_SCALAR (PokerEnv.py:361-368) */
    double norm;           /* observation normaliser = mean starting stack (PokerEnv.py:1267) */
} prl_env_cfg_t;

/* number of int32 state fields per table; state = DEVICE int32[prl_env_state_fields()][n_envs] */
int prl_env_state_fields(void);

/* PokerEnv.reset (PokerEnv.py:1075-1122) for all tables.  deck = DEVICE int8[n_envs][n_deck], top card first: seat 0's
 * hole cards, seat 1's, flop, turn, river (_Deck.py:23-27).  shuffle != 0 fills the decks from a counter RNG
 * (seed, episode0 + table) instead of using the caller's.  obs = DEVICE float[n_envs][obs_size] or NULL,
 * legal = DEVICE uint8[n_envs][n_actions] or NULL (get_legal_actions as a mask). */
int prl_env_reset(const prl_env_cfg_t* cfg, int32_t* state, int8_t* deck, float* obs, uint8_t* legal, uint64_t seed,
                  uint64_t episode0, int shuffle, prl_stream_t stream);

/* PokerEnv.step (PokerEnv.py:1148-1159, 681-789) for all tables: actions = DEVICE int32[n_envs] discrete actions, or
 * NULL / negative entries = uniformly random legal action from the counter RNG (seed, step_id).  Outputs (any may be
 * NULL): obs (zeros at terminal states), rewards = DEVICE double[n_envs][2] ((stack - start) / REWARD_SCALAR at terminal
 * steps, else 0), done = DEVICE uint8[n_envs], legal mask for the next step.  Finished tables ignore further steps unless
 * auto_reset != 0, in which case they are re-dealt (counter RNG) and reset before the action is applied. */
int prl_env_step(const prl_env_cfg_t* cfg, int32_t* state, int8_t* deck, const int32_t* actions, float* obs,
                 double* rewards, uint8_t* done, uint8_t* legal, uint64_t seed, uint64_t step_id, int auto_reset,
                 prl_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Head-to-head play of two tabular agents (replaces the per-hand loop of
 * PokerRL/eval/head_to_head/LocalHead2HeadMaster.py:81-126).  One table of the batched env per hand; each table walks
 * the agents' shared public tree in step with its env.  Hands [0, n_hands_per_seat) have agent A in seat 0, the rest
 * agent A in seat 1.  Host loop: prl_h2h_step, then prl_env_step with the actions it wrote, at most "tree depth" times,
 * one more prl_h2h_step, then prl_h2h_collect.
 * ------------------------------------------------------------------------------------------------------------------ */
typedef struct {
    int32_t n_envs;           /* tables in this batch (= prl_env_cfg_t.n_envs) */
    int32_t n_range;          /* hands per seat (RANGE_SIZE) */
    int32_t n_hole;           /* 1: hand = card, chance child = rank of the dealt card among the cards not on the board;
                                 2: hand = lexicographic index of (c1 < c2) */
    int32_t chance_by_class;  /* 1: chance child = board_class[lexicographic rank of the sorted 5-card board] */
    int32_t max_decisions;    /* row width of `uniforms` */
    int64_t seat_swap_at;     /* global hands >= this one have agent A in seat 1 */
    int64_t hand0;            /* global index of this batch's first hand (counter RNG, seat assignment) */
    uint64_t seed;
    const int8_t* kind;       /* DEVICE int8[n_nodes]  flat tree (game/flat_tree.py) */
    const int32_t* first_child, *n_children, *first_slot, *action;
    const float* table_a;     /* DEVICE float32[n_slots][ld_a]: agent A's action probabilities */
    const float* table_b;
    int64_t ld_a, ld_b;
    const int32_t* board_class; /* DEVICE int32[C(52,5)] or NULL */
    const uint8_t* board_perm;  /* DEVICE uint8[C(52,5)]: suit permutation s mapping the board onto its class */
    const int16_t* sym_perm;    /* DEVICE int16[24][n_range]: hand h on the board reads row sym_perm[s][h] */
    const double* uniforms;     /* DEVICE float64[n_envs][max_decisions] (replays) or NULL: counter RNG (seed, hand, k) */
    int32_t* node;            /* DEVICE int32[n_envs]  per-table tree node, -1 after a desync */
    int32_t* n_dec;           /* DEVICE int32[n_envs]  decisions taken so far */
    uint8_t* perm;            /* DEVICE uint8[n_envs]  suit permutation of the dealt board */
    int32_t* chips;           /* DEVICE int32[n_envs]  agent A's chip result once the hand ended */
    unsigned long long* desync; /* DEVICE uint64[1]    invariant violations (acting seat / terminal state) */
} prl_h2h_t;

/* Starts every table at the root (node 0, no decision taken). */
int prl_h2h_init(const prl_h2h_t* h, int32_t* actions, prl_stream_t stream);

/* Moves each table's node by actions[i] (the action the env just applied) and through a chance node by the dealt board,
 * checks the node against the env (state / deck / rewards of prl_env_step), and writes the next action of a table whose
 * node is a decision node, sampled like EvalAgentBase.get_action; -1 where the hand is over. */
int prl_h2h_step(const prl_h2h_t* h, const prl_env_cfg_t* cfg, const int32_t* state, const int8_t* deck,
                 const double* rewards, int32_t* actions, prl_stream_t stream);

/* Tables whose node is not terminal here (a hand the loop did not finish) count as desyncs.
 * sums[0] += sum of agent A's chip results, sums[1] += sum of their squares (DEVICE int64[2]); winnings = DEVICE
 * float32[n_envs] or NULL: chips / REWARD_SCALAR * REWARD_SCALAR * ev_normalizer per hand. */
int prl_h2h_collect(const prl_h2h_t* h, double reward_scalar, double ev_normalizer, long long* sums, float* winnings,
                    prl_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* POKERRL_B200_H */
