// Head-to-head play of two tabular agents on the batched env (sm_100a), one thread per table.
//
// Restates the hand loop of PokerRL/eval/head_to_head/LocalHead2HeadMaster.py:81-126 for n tables in lockstep: each
// table carries the node of the agents' shared public tree (game/flat_tree.py) it has reached, moves it by the action the
// env applied and through a chance node by the board the env dealt, and samples the acting agent's next action from that
// node's rows of the agent's table with the rule of EvalAgentBase.get_action (float64 cumulative sum in action order,
// first entry above the uniform, else the last action with mass).  The env (csrc/env_kernels.cu) keeps doing all game
// logic; this file only reads its state, so a tree that disagrees with the env is counted, never followed.
//
// Chips are integers, so the sums of agent A's results and of their squares are int64 and do not depend on the grid or
// on how hands are split into batches.
#include <cuda_runtime.h>
#include <stdint.h>

#include "env_state.cuh"
#include "pokerrl_b200.h"
#include "prl_common.cuh"

namespace {

using namespace prl_env;

constexpr int kThreads = 128;

__host__ __device__ __forceinline__ uint64_t splitmix64(uint64_t z) {
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

// uniform of decision k of global hand g: 53 random bits in [0, 1) (restated by eval/head_to_head/match.counter_uniforms)
__device__ __forceinline__ double counter_uniform(uint64_t seed, uint64_t g, uint64_t k) {
    const uint64_t x = splitmix64(splitmix64(seed ^ splitmix64(g)) + k);
    return (double)(x >> 11) * 0x1.0p-53;
}

__device__ __forceinline__ int64_t binom_small(int n, int k) {  // C(n, k) for k <= 5, 0 if n < k
    if (n < k) return 0;
    int64_t r = 1;
    for (int i = 0; i < k; ++i) r = r * (n - i) / (i + 1);
    return r;
}

// lexicographic rank of a sorted 5-card board among all C(52, 5) (the order of holdem_boards._combos_52_5)
__device__ __forceinline__ int board_rank_52_5(const int* c) {
    int64_t colex = 0;
    for (int i = 0; i < 5; ++i) colex += binom_small(51 - c[i], 5 - i);
    return (int)(2598959ll - colex);
}

__device__ __forceinline__ int cards_out_at(const prl_env_cfg_t& g, int round) {
    return (round >= 1 ? g.n_flop : 0) + (round >= 2 ? g.n_turn : 0) + (round >= 3 ? g.n_river : 0);
}

// child of chance node n for the board in the deck (round = the env's round after the deal); -1 if it cannot be read
__device__ int chance_child(const prl_h2h_t& h, const prl_env_cfg_t& g, int n, const int8_t* d, int round, uint8_t& perm) {
    const int8_t* board = d + 2 * g.n_hole;
    int j;
    if (h.chance_by_class) {
        int c[5];
        for (int i = 0; i < 5; ++i) c[i] = board[i];
        for (int i = 1; i < 5; ++i)  // insertion sort
            for (int k = i; k > 0 && c[k - 1] > c[k]; --k) { const int t = c[k]; c[k] = c[k - 1]; c[k - 1] = t; }
        const int r = board_rank_52_5(c);
        j = h.board_class[r];
        perm = h.board_perm[r];
    } else {  // one new card: rank among the cards not on the board before the deal (flat_tree.make_board_tables)
        const int n_prev = cards_out_at(g, round - 1);
        if (cards_out_at(g, round) != n_prev + 1) return -1;
        const int card = board[n_prev];
        j = card;
        for (int i = 0; i < n_prev; ++i) j -= (board[i] < card) ? 1 : 0;
    }
    return (j >= 0 && j < h.n_children[n]) ? h.first_child[n] + j : -1;
}

__global__ void __launch_bounds__(kThreads) h2h_init_kernel(prl_h2h_t h, int32_t* actions) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= h.n_envs) return;
    h.node[i] = 0;
    h.n_dec[i] = 0;
    h.perm[i] = 0;
    h.chips[i] = 0;
    actions[i] = -1;
}

__global__ void __launch_bounds__(kThreads) h2h_step_kernel(prl_h2h_t h, prl_env_cfg_t g, const int32_t* st, const int8_t* deck,
                                                            const double* rew, int32_t* actions) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int B = h.n_envs;
    if (i >= B) return;
    int node = h.node[i];
    const bool done = st[F_DONE * B + i] != 0;
    if (node < 0) {  // desynced earlier: let the env finish the hand without following it
        actions[i] = done ? -1 : 0;
        return;
    }
    const int64_t gh = h.hand0 + i;
    const int a_seat = gh >= h.seat_swap_at ? 1 : 0;
    const int8_t* d = deck + (size_t)i * g.n_deck;
    const int a = actions[i];
    bool ok = true;
    if (a >= 0) {  // the env applied action a at this node
        const int fc = h.first_child[node], nc = h.n_children[node];
        int child = -1;
        if (h.kind[node] <= PRL_KIND_P1)
            for (int k = 0; k < nc; ++k)
                if (h.action[fc + k] == a) child = fc + k;
        node = child;
        if (node >= 0 && h.kind[node] == PRL_KIND_CHANCE) {
            uint8_t p = h.perm[i];
            node = chance_child(h, g, node, d, st[F_ROUND * B + i], p);
            h.perm[i] = p;
        }
        ok = node >= 0;
    }
    int next = -1;
    if (ok) {
        const int kd = h.kind[node];
        if (done) {
            ok = kd >= PRL_KIND_FOLD;
            if (ok && a >= 0) h.chips[i] = (int32_t)llrint(rew[2 * (size_t)i + a_seat] * g.reward_scalar);
        } else {
            ok = kd <= PRL_KIND_P1 && kd == st[F_CUR * B + i];
        }
        if (ok && !done) {
            const int k = h.n_dec[i];
            h.n_dec[i] = k + 1;
            double u;
            if (h.uniforms) {
                ok = k < h.max_decisions;
                u = ok ? h.uniforms[(size_t)i * h.max_decisions + k] : 0.0;
            } else {
                u = counter_uniform(h.seed, (uint64_t)gh, (uint64_t)k);
            }
            const int8_t* hole = d + kd * g.n_hole;
            int hand = hole[0];
            if (h.n_hole == 2) {
                const int c1 = min(hole[0], hole[1]), c2 = max(hole[0], hole[1]);
                hand = c1 * (2 * g.n_deck - c1 - 1) / 2 + (c2 - c1 - 1);
            }
            if (h.chance_by_class) hand = h.sym_perm[(size_t)h.perm[i] * h.n_range + hand];
            const bool is_a = kd == a_seat;
            const float* tab = is_a ? h.table_a : h.table_b;
            const int64_t ld = is_a ? h.ld_a : h.ld_b;
            const int fs = h.first_slot[node], fc = h.first_child[node], nc = h.n_children[node];
            double cum = 0.0;
            int pick = -1, last_mass = -1;
            for (int j = 0; j < nc; ++j) {
                const float p = tab[(size_t)(fs + j) * ld + hand];
                cum += (double)p;
                if (p != 0.0f) last_mass = j;
                if (pick < 0 && cum > u) pick = j;
            }
            if (pick < 0) pick = last_mass;  // the draw fell beyond the last action with mass through rounding
            next = pick >= 0 ? h.action[fc + pick] : 0;
        }
    }
    if (!ok) {
        atomicAdd(h.desync, 1ull);
        node = -1;
        next = done ? -1 : 0;
    }
    h.node[i] = node;
    actions[i] = next;
}

__global__ void __launch_bounds__(kThreads) h2h_collect_kernel(prl_h2h_t h, double reward_scalar, double ev_normalizer,
                                                               long long* sums, float* winnings) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    long long w = 0;
    if (i < h.n_envs) {
        const int n = h.node[i];
        if (n >= 0 && h.kind[n] < PRL_KIND_FOLD) atomicAdd(h.desync, 1ull);  // the hand did not finish in the loop
        w = h.chips[i];
        if (winnings) winnings[i] = (float)((double)w / reward_scalar * reward_scalar * ev_normalizer);
    }
    long long s = w, q = w * w;
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_down_sync(0xffffffffu, s, o);
        q += __shfl_down_sync(0xffffffffu, q, o);
    }
    __shared__ long long red[2][kThreads / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) { red[0][warp] = s; red[1][warp] = q; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 1; k < kThreads / 32; ++k) { s += red[0][k]; q += red[1][k]; }
        atomicAdd((unsigned long long*)&sums[0], (unsigned long long)s);
        atomicAdd((unsigned long long*)&sums[1], (unsigned long long)q);
    }
}

int check_h2h(const prl_h2h_t* h) {
    if (!h || h->n_envs <= 0) return prl::fail("prl_h2h: bad batch");
    if (!h->kind || !h->first_child || !h->n_children || !h->first_slot || !h->action || !h->table_a || !h->table_b)
        return prl::fail("prl_h2h: tree or table pointer missing");
    if (!h->node || !h->n_dec || !h->perm || !h->chips || !h->desync) return prl::fail("prl_h2h: per-table buffer missing");
    if (h->n_hole != 1 && h->n_hole != 2) return prl::fail("prl_h2h: n_hole must be 1 or 2");
    if (h->chance_by_class && (!h->board_class || !h->board_perm || !h->sym_perm || h->n_hole != 2))
        return prl::fail("prl_h2h: chance_by_class needs board_class / board_perm / sym_perm of a two-card game");
    if (h->uniforms && h->max_decisions <= 0) return prl::fail("prl_h2h: uniforms need max_decisions > 0");
    return 0;
}

inline int grid(int n) { return (n + kThreads - 1) / kThreads; }

}  // namespace

extern "C" int prl_h2h_init(const prl_h2h_t* h, int32_t* actions, prl_stream_t stream) {
    if (int e = check_h2h(h)) return e;
    h2h_init_kernel<<<grid(h->n_envs), kThreads, 0, (cudaStream_t)stream>>>(*h, actions);
    prl::count_launch();
    return prl::check(cudaGetLastError(), "prl_h2h_init");
}

extern "C" int prl_h2h_step(const prl_h2h_t* h, const prl_env_cfg_t* cfg, const int32_t* state, const int8_t* deck,
                            const double* rewards, int32_t* actions, prl_stream_t stream) {
    if (int e = check_h2h(h)) return e;
    if (!cfg || cfg->n_envs != h->n_envs || cfg->n_hole != h->n_hole) return prl::fail("prl_h2h_step: env config mismatch");
    h2h_step_kernel<<<grid(h->n_envs), kThreads, 0, (cudaStream_t)stream>>>(*h, *cfg, state, deck, rewards, actions);
    prl::count_launch();
    return prl::check(cudaGetLastError(), "prl_h2h_step");
}

extern "C" int prl_h2h_collect(const prl_h2h_t* h, double reward_scalar, double ev_normalizer, long long* sums,
                               float* winnings, prl_stream_t stream) {
    if (int e = check_h2h(h)) return e;
    h2h_collect_kernel<<<grid(h->n_envs), kThreads, 0, (cudaStream_t)stream>>>(*h, reward_scalar, ev_normalizer, sums,
                                                                               winnings);
    prl::count_launch();
    return prl::check(cudaGetLastError(), "prl_h2h_collect");
}
