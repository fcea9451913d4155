// Batched heads-up PokerEnv: reset / step for B independent tables, one thread per table (sm_100a).
//
// Restates the reference's scalar Python engine for two seats (SURVEY.md appendix B), integer chip accounting:
//   reset            PokerRL/game/_/rl_env/base/PokerEnv.py:1075-1122        legalisation  PokerEnv.py:885-941
//   step / apply     PokerEnv.py:681-732                                     round end     PokerEnv.py:943-954
//   transitions      PokerEnv.py:737-789, rundown :620-644, payout :471-531  min raise     PokerEnv.py:809-812
//   pot fraction     PokerEnv.py:1376-1396                                   observation   PokerEnv.py:1004-1031, 964-1002, 1253-1271
//   discretized      poker_types/DiscretizedPokerEnv.py:44-135               limit         poker_types/LimitPokerEnv.py:27-59, games.py:253-254
//   deck             base/_Deck.py:20-31 (cards are drawn from the top, seat 0 first, then flop / turn / river)
// The same transition function is implemented on the host by pokerrl_b200/game/hu_engine.py (tree compiler).
// Parity: tests/test_gpu_env.py replays decks + actions recorded from the reference env (tests/golden/env_*.npz) and
// requires identical observations, rewards, done flags and legal-action masks.
//
// Table state is SoA int32[kFields][B] (coalesced across tables); observations are written row-major float32[B][obs].
#include <cuda_runtime.h>
#include <stdint.h>

#include "env_state.cuh"
#include "hand_eval.cuh"
#include "pokerrl_b200.h"
#include "prl_common.cuh"

namespace {

using namespace prl_env;
enum { FL_ALLIN0 = 1, FL_ALLIN1 = 2, FL_FOLD0 = 4, FL_FOLD1 = 8, FL_ACTED0 = 16, FL_ACTED1 = 32 };
enum { FOLD = 0, CALL = 1, RAISE = 2 };

struct Table {
    int round, pot, stack[2], bet[2], flags, cur, last_raiser, n_act_ep, n_raises, capped, cap_raiser, cap_noreopen;
    int last_type, last_amt, last_who, done;
    __device__ bool allin(int p) const { return flags & (FL_ALLIN0 << p); }
    __device__ bool folded(int p) const { return flags & (FL_FOLD0 << p); }
    __device__ bool acted(int p) const { return flags & (FL_ACTED0 << p); }
};

__device__ __forceinline__ void load_table(const int32_t* st, int B, int i, Table& t) {
    t.round = st[F_ROUND * B + i];
    t.pot = st[F_POT * B + i];
    t.stack[0] = st[F_STACK0 * B + i];
    t.stack[1] = st[F_STACK1 * B + i];
    t.bet[0] = st[F_BET0 * B + i];
    t.bet[1] = st[F_BET1 * B + i];
    t.flags = st[F_FLAGS * B + i];
    t.cur = st[F_CUR * B + i];
    t.last_raiser = st[F_LAST_RAISER * B + i];
    t.n_act_ep = st[F_N_ACT_EP * B + i];
    t.n_raises = st[F_N_RAISES * B + i];
    t.capped = st[F_CAPPED * B + i];
    t.cap_raiser = st[F_CAP_RAISER * B + i];
    t.cap_noreopen = st[F_CAP_NOREOPEN * B + i];
    t.last_type = st[F_LAST_TYPE * B + i];
    t.last_amt = st[F_LAST_AMT * B + i];
    t.last_who = st[F_LAST_WHO * B + i];
    t.done = st[F_DONE * B + i];
}

__device__ __forceinline__ void store_table(int32_t* st, int B, int i, const Table& t) {
    st[F_ROUND * B + i] = t.round;
    st[F_POT * B + i] = t.pot;
    st[F_STACK0 * B + i] = t.stack[0];
    st[F_STACK1 * B + i] = t.stack[1];
    st[F_BET0 * B + i] = t.bet[0];
    st[F_BET1 * B + i] = t.bet[1];
    st[F_FLAGS * B + i] = t.flags;
    st[F_CUR * B + i] = t.cur;
    st[F_LAST_RAISER * B + i] = t.last_raiser;
    st[F_N_ACT_EP * B + i] = t.n_act_ep;
    st[F_N_RAISES * B + i] = t.n_raises;
    st[F_CAPPED * B + i] = t.capped;
    st[F_CAP_RAISER * B + i] = t.cap_raiser;
    st[F_CAP_NOREOPEN * B + i] = t.cap_noreopen;
    st[F_LAST_TYPE * B + i] = t.last_type;
    st[F_LAST_AMT * B + i] = t.last_amt;
    st[F_LAST_WHO * B + i] = t.last_who;
    st[F_DONE * B + i] = t.done;
}

// ---- primitives (PokerPlayer.bet_raise / check_call, _put_current_bets_into_main_pot_and_side_pots) -------------------
__device__ __forceinline__ void bet_to(Table& t, int p, int total) {
    t.flags |= FL_ACTED0 << p;
    t.stack[p] -= total - t.bet[p];
    t.bet[p] = total;
    if (t.stack[p] == 0) t.flags |= FL_ALLIN0 << p;
}

__device__ __forceinline__ void bets_into_pot(Table& t) {
    const int d = t.bet[0] - t.bet[1];
    if (d > 0) { t.stack[0] += d; t.bet[0] -= d; }
    else if (d < 0) { t.stack[1] -= d; t.bet[1] += d; }
    t.pot += t.bet[0] + t.bet[1];
    t.bet[0] = t.bet[1] = 0;
}

__device__ __forceinline__ int min_raise_total(const prl_env_cfg_t& g, const Table& t) {
    const int lo = min(t.bet[0], t.bet[1]), hi = max(t.bet[0], t.bet[1]);
    return hi + max(hi - lo, g.big_blind);
}

__device__ __forceinline__ int pot_fraction_raise(const Table& t, double frac, int p) {
    const int to_call = max(t.bet[0], t.bet[1]) - t.bet[p];
    const int pot_after_call = t.pot + t.bet[0] + t.bet[1] + to_call;
    return (int)((double)to_call + (double)pot_after_call * frac) + t.bet[p];  // int() truncation of a float64 product
}

__device__ __forceinline__ void decode(const prl_env_cfg_t& g, const Table& t, int a, int& typ, int& chips) {
    if (a == FOLD) { typ = FOLD; chips = -1; }
    else if (a == CALL) { typ = CALL; chips = -1; }
    else if (g.kind == 1) { typ = RAISE; chips = pot_fraction_raise(t, g.fracs[a - 2], t.cur); }
    else { typ = RAISE; chips = -1; }
}

__device__ __forceinline__ int adjust_raise(const prl_env_cfg_t& g, const Table& t, int chips) {
    if (g.kind == 0) {
        if (g.limit_raise_is_pot) return pot_fraction_raise(t, 1.0, t.cur);
        const int b = (t.round >= g.round_big_bet_starts) ? g.big_bet : g.small_bet;
        return (t.n_raises + 1) * b;
    }
    return max(min_raise_total(g, t), chips);
}

// PokerEnv._get_fixed_action
__device__ __forceinline__ void fix_action(const prl_env_cfg_t& g, const Table& t, int typ, int chips, int& ftyp, int& famt) {
    const int p = t.cur;
    const int total_to_call = max(t.bet[0], t.bet[1]);
    const int call_amt = min(total_to_call - t.bet[p], t.stack[p]) + t.bet[p];
    if (typ == FOLD) {
        if (total_to_call <= t.bet[p]) { ftyp = CALL; famt = call_amt; }
        else { ftyp = FOLD; famt = -1; }
        return;
    }
    if (typ == CALL) {
        if (g.first_action_no_call && t.n_act_ep == 0 && t.round == 0) { ftyp = FOLD; famt = -1; }
        else { ftyp = CALL; famt = call_amt; }
        return;
    }
    if (g.kind == 0 && t.n_raises >= g.max_raises[t.round]) { ftyp = CALL; famt = call_amt; return; }
    if (t.stack[p] + t.bet[p] <= total_to_call || (t.capped && t.cap_noreopen == p)) { ftyp = CALL; famt = call_amt; return; }
    int raise_to = adjust_raise(g, t, chips);
    if (t.bet[p] + t.stack[p] < raise_to) raise_to = t.stack[p] + t.bet[p];
    ftyp = RAISE;
    famt = raise_to;
}

// get_legal_actions (DiscretizedPokerEnv.py:99-135, LimitPokerEnv.py:41-59) as a mask over the discrete actions
__device__ void legal_mask(const prl_env_cfg_t& g, const Table& t, uint8_t* mask) {
    for (int a = 0; a < g.n_actions; ++a) mask[a] = 0;
    if (t.done) return;
    int ft, fa;
    fix_action(g, t, FOLD, -1, ft, fa);
    if (ft == FOLD) mask[FOLD] = 1;
    fix_action(g, t, CALL, -1, ft, fa);
    if (ft == CALL) mask[CALL] = 1;
    if (g.kind == 0) {
        fix_action(g, t, RAISE, -1, ft, fa);
        if (t.n_raises < g.max_raises[t.round] && ft == RAISE) mask[RAISE] = 1;
        return;
    }
    int last_too_small = -1;
    for (int a = 2; a < g.n_actions; ++a) {
        int typ, want;
        decode(g, t, a, typ, want);
        fix_action(g, t, typ, want, ft, fa);
        if (ft != typ) break;
        if (want < fa) {
            last_too_small = a;
        } else {
            if (last_too_small >= 0) { mask[last_too_small] = 1; last_too_small = -1; }
            mask[a] = 1;
        }
        if (want > fa) break;
    }
}

// ---- cards --------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int cards_out_at(const prl_env_cfg_t& g, int round) {
    return (round >= 1 ? g.n_flop : 0) + (round >= 2 ? g.n_turn : 0) + (round >= 3 ? g.n_river : 0);
}

// strength of seat p's hand with the full board (PokerEnv._assign_hand_ranks_to_all_players)
__device__ int hand_strength(const prl_env_cfg_t& g, const int8_t* deck, int p) {
    const int8_t* hole = deck + p * g.n_hole;
    const int8_t* board = deck + 2 * g.n_hole;
    if (g.n_hole == 1) {  // Leduc family (game_rules.py:68-75, 134-141)
        const int r = hole[0] / g.n_suits;
        return (board[0] / g.n_suits == r) ? g.pair_bonus + r : r;
    }
    prl_he::CardSet cs = {0ull, {0u, 0u, 0u, 0u}};
    cs.add(hole[0]);
    cs.add(hole[1]);
    for (int i = 0; i < 5; ++i) cs.add(board[i]);
    return prl_he::rank_cardset(cs);
}

// ---- observation (PokerEnv.get_current_obs for the simplified heads-up layout) -------------------------------------------
__device__ void write_obs(const prl_env_cfg_t& g, const Table& t, const int8_t* deck, float* obs) {
    const int n = g.obs_size;
    for (int k = 0; k < n; ++k) obs[k] = 0.0f;
    if (t.done) return;  // terminal observation is all zeros (PokerEnv.py:1265-1266)
    const double norm = g.norm;
    int k = 0;
    obs[k++] = (float)((double)g.ante / norm);
    obs[k++] = (float)((double)g.small_blind / norm);
    obs[k++] = (float)((double)g.big_blind / norm);
    obs[k++] = (float)((double)min_raise_total(g, t) / norm);
    obs[k++] = (float)((double)t.pot / norm);
    obs[k++] = (float)((double)max(t.bet[0], t.bet[1]) / norm);
    obs[k++] = (t.last_type >= 0) ? (float)((double)t.last_amt / norm) : 0.0f;
    if (t.last_type >= 0) {
        obs[k + t.last_type] = 1.0f;
        obs[k + 3 + t.last_who] = 1.0f;
    }
    k += 5;
    obs[k + t.cur] = 1.0f;
    k += 2;
    obs[k + t.round] = 1.0f;
    k += g.n_round_slots;
    for (int p = 0; p < 2; ++p) {
        obs[k++] = (float)((double)t.stack[p] / norm);
        obs[k++] = (float)((double)t.bet[p] / norm);
        obs[k++] = t.allin(p) ? 1.0f : 0.0f;
    }
    const int per = g.n_ranks + g.n_suits;
    const int n_out = cards_out_at(g, t.round);
    const int8_t* board = deck + 2 * g.n_hole;
    for (int i = 0; i < n_out; ++i) {
        const int c = board[i];
        obs[k + per * i + c / g.n_suits] = 1.0f;
        if (g.suits_matter) obs[k + per * i + g.n_ranks + c % g.n_suits] = 1.0f;
    }
}

// ---- reset / step ---------------------------------------------------------------------------------------------------
__device__ void reset_table(const prl_env_cfg_t& g, Table& t) {
    t.n_raises = (g.kind == 0) ? (g.big_blind > 0 ? 1 : 0) : 0;
    t.pot = 0;
    t.round = 0;
    t.capped = 0;
    t.cap_raiser = t.cap_noreopen = -1;
    t.last_raiser = -1;
    t.n_act_ep = 0;
    t.last_type = t.last_amt = t.last_who = -1;
    t.stack[0] = g.start_stack[0];
    t.stack[1] = g.start_stack[1];
    t.bet[0] = t.bet[1] = 0;
    t.flags = 0;
    t.done = 0;
    bet_to(t, 0, g.ante);  // antes go straight into the pot (PokerEnv.py:1111-1112)
    bet_to(t, 1, g.ante);
    bets_into_pot(t);
    bet_to(t, 0, g.small_blind);  // heads-up: seat 0 = button = small blind (PokerEnv.py:337-340)
    bet_to(t, 1, g.big_blind);
    t.flags &= ~(FL_ACTED0 | FL_ACTED1);
    t.cur = 0;
}

__device__ void award_showdown(const prl_env_cfg_t& g, Table& t, const int8_t* deck, double* stack_out) {
    // bets are already in the pot; higher strength takes it, a tie splits it (PokerEnv.py:471-481)
    const int r0 = hand_strength(g, deck, 0), r1 = hand_strength(g, deck, 1);
    stack_out[0] = (double)t.stack[0];
    stack_out[1] = (double)t.stack[1];
    if (r0 > r1) stack_out[0] += (double)t.pot;
    else if (r0 < r1) stack_out[1] += (double)t.pot;
    else { stack_out[0] += (double)t.pot / 2.0; stack_out[1] += (double)t.pot / 2.0; }
}

__device__ void step_table(const prl_env_cfg_t& g, Table& t, const int8_t* deck, int action, double* rew) {
    rew[0] = rew[1] = 0.0;
    if (t.done) return;
    int typ, chips, ftyp, famt;
    decode(g, t, action, typ, chips);
    fix_action(g, t, typ, chips, ftyp, famt);
    const int p = t.cur;
    if (ftyp == CALL) {
        bet_to(t, p, famt);
    } else if (ftyp == FOLD) {
        t.flags |= (FL_ACTED0 << p) | (FL_FOLD0 << p);
    } else {
        if (famt < min_raise_total(g, t)) {  // under-min all-in: the previous raiser may not re-open (PokerEnv.py:710-714)
            t.capped = 1;
            t.cap_raiser = p;
            t.cap_noreopen = t.last_raiser;
        } else if (t.capped && t.cap_noreopen != p) {
            t.capped = 0;
            t.cap_raiser = t.cap_noreopen = -1;
        }
        t.last_raiser = p;
        bet_to(t, p, famt);
        t.n_act_ep += 1;
        if (g.kind == 0) t.n_raises += 1;
    }
    t.last_type = ftyp;
    t.last_amt = famt;
    t.last_who = p;

    const int n_nonfold = (t.folded(0) ? 0 : 1) + (t.folded(1) ? 0 : 1);
    const bool live0 = !t.folded(0) && !t.allin(0), live1 = !t.folded(1) && !t.allin(1);
    const int n_live = (live0 ? 1 : 0) + (live1 ? 1 : 0);
    bool cont = false;
    if (n_nonfold >= 2) {  // PokerEnv._should_continue_in_this_round
        const int largest = max(t.bet[0], t.bet[1]);
        const bool settled = (t.folded(0) || t.allin(0) || t.bet[0] == largest) && (t.folded(1) || t.allin(1) || t.bet[1] == largest);
        const bool all_acted = (!live0 || t.acted(0)) && (!live1 || t.acted(1));
        cont = !(settled && all_acted);
    }
    double final_stack[2];
    bool terminal = false;
    if (cont) {
        const int q = 1 - p;
        t.cur = (!t.allin(q) && !t.folded(q)) ? q : p;
    } else if (n_live > 1) {
        if (t.round == g.n_rounds - 1) {
            bets_into_pot(t);
            award_showdown(g, t, deck, final_stack);
            terminal = true;
        } else {  // PokerEnv._next_round
            if (g.kind == 0) t.n_raises = 0;
            t.capped = 0;
            t.cap_raiser = t.cap_noreopen = -1;
            bets_into_pot(t);
            t.cur = g.btn_first_postflop ? 0 : 1;
            t.flags &= ~(FL_ACTED0 | FL_ACTED1);
            t.round += 1;
        }
    } else if (n_nonfold > 1) {  // someone is all-in: run the board out and pay (PokerEnv._rundown)
        bets_into_pot(t);
        t.round = g.n_rounds - 1;
        award_showdown(g, t, deck, final_stack);
        terminal = true;
    } else {  // everybody else folded: PokerEnv._pay_all_to_one_player
        const int w = t.folded(0) ? 1 : 0;
        final_stack[0] = (double)t.stack[0];
        final_stack[1] = (double)t.stack[1];
        final_stack[w] += (double)(t.bet[0] + t.bet[1] + t.pot);
        t.bet[0] = t.bet[1] = 0;
        terminal = true;
    }
    if (terminal) {
        t.done = 1;
        rew[0] = (final_stack[0] - (double)g.start_stack[0]) / g.reward_scalar;  // PokerEnv.py:1069-1072
        rew[1] = (final_stack[1] - (double)g.start_stack[1]) / g.reward_scalar;
        t.stack[0] = (int)final_stack[0];
        t.stack[1] = (int)final_stack[1];
        t.pot = 0;
    }
}

// ---- counter-based RNG (deck shuffles and uniform legal actions for the throughput workload) -----------------------------
__device__ __forceinline__ uint32_t mix32(uint64_t x) {  // splitmix64 finaliser
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return (uint32_t)((x ^ (x >> 31)) >> 16);
}

__device__ void shuffle_deck(int8_t* deck, int n_deck, uint64_t seed, uint64_t stream) {
    for (int c = 0; c < n_deck; ++c) deck[c] = (int8_t)c;
    for (int i = n_deck - 1; i > 0; --i) {  // Fisher-Yates
        const int j = (int)(mix32(seed ^ (stream * 0x100000001B3ull + (uint64_t)i)) % (uint32_t)(i + 1));
        const int8_t tmp = deck[i];
        deck[i] = deck[j];
        deck[j] = tmp;
    }
}

__global__ void __launch_bounds__(128) env_reset_kernel(prl_env_cfg_t g, int32_t* state, int8_t* deck, float* obs, uint8_t* legal,
                                                        uint64_t seed, uint64_t episode0, int shuffle) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= g.n_envs) return;
    int8_t* d = deck + (size_t)i * g.n_deck;
    if (shuffle) shuffle_deck(d, g.n_deck, seed, episode0 + (uint64_t)i);
    Table t;
    reset_table(g, t);
    store_table(state, g.n_envs, i, t);
    if (obs) write_obs(g, t, d, obs + (size_t)i * g.obs_size);
    if (legal) legal_mask(g, t, legal + (size_t)i * g.n_actions);
}

// action < 0: sample uniformly among the legal actions (counter RNG); auto_reset: finished tables start a new hand
__global__ void __launch_bounds__(128) env_step_kernel(prl_env_cfg_t g, int32_t* state, int8_t* deck, const int32_t* actions,
                                                       float* obs, double* rew, uint8_t* done, uint8_t* legal, uint64_t seed,
                                                       uint64_t step_id, int auto_reset) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= g.n_envs) return;
    int8_t* d = deck + (size_t)i * g.n_deck;
    Table t;
    load_table(state, g.n_envs, i, t);
    if (t.done && auto_reset) {
        shuffle_deck(d, g.n_deck, seed, (step_id << 24) ^ (uint64_t)i ^ 0xABCDEF12345ull);
        reset_table(g, t);
    }
    int a = actions ? actions[i] : -1;
    if (a < 0 && !t.done) {
        uint8_t m[PRL_ENV_MAX_ACTIONS];
        legal_mask(g, t, m);
        int n = 0;
        for (int k = 0; k < g.n_actions; ++k) n += m[k];
        int pick = (int)(mix32(seed ^ (step_id * 0x9E3779B1ull) ^ ((uint64_t)i << 20)) % (uint32_t)max(n, 1));
        for (int k = 0; k < g.n_actions; ++k)
            if (m[k] && pick-- == 0) { a = k; break; }
    }
    double r[2];
    step_table(g, t, d, a, r);
    store_table(state, g.n_envs, i, t);
    if (obs) write_obs(g, t, d, obs + (size_t)i * g.obs_size);
    if (rew) { rew[2 * (size_t)i] = r[0]; rew[2 * (size_t)i + 1] = r[1]; }
    if (done) done[i] = (uint8_t)t.done;
    if (legal) legal_mask(g, t, legal + (size_t)i * g.n_actions);
}

int check_cfg(const prl_env_cfg_t* g) {
    if (!g || g->n_envs <= 0) return prl::fail("prl_env: bad config");
    if (g->n_actions > PRL_ENV_MAX_ACTIONS || g->n_actions < 3) return prl::fail("prl_env: n_actions out of range");
    if (g->n_hole < 1 || g->n_hole > 2 || g->n_deck > 52) return prl::fail("prl_env: unsupported deck / hand size");
    return 0;
}

}  // namespace

extern "C" int prl_env_state_fields(void) { return kFields; }

extern "C" int prl_env_reset(const prl_env_cfg_t* cfg, int32_t* state, int8_t* deck, float* obs, uint8_t* legal,
                             uint64_t seed, uint64_t episode0, int shuffle, prl_stream_t stream) {
    if (int e = check_cfg(cfg)) return e;
    env_reset_kernel<<<(cfg->n_envs + 127) / 128, 128, 0, (cudaStream_t)stream>>>(*cfg, state, deck, obs, legal, seed, episode0, shuffle);
    prl::count_launch();
    return prl::check(cudaGetLastError(), "prl_env_reset");
}

extern "C" int prl_env_step(const prl_env_cfg_t* cfg, int32_t* state, int8_t* deck, const int32_t* actions, float* obs,
                            double* rewards, uint8_t* done, uint8_t* legal, uint64_t seed, uint64_t step_id, int auto_reset,
                            prl_stream_t stream) {
    if (int e = check_cfg(cfg)) return e;
    env_step_kernel<<<(cfg->n_envs + 127) / 128, 128, 0, (cudaStream_t)stream>>>(*cfg, state, deck, actions, obs, rewards, done,
                                                                                 legal, seed, step_id, auto_reset);
    prl::count_launch();
    return prl::check(cudaGetLastError(), "prl_env_step");
}
