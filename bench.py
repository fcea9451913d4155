"""Benchmark of the CFR hot path (BASELINE.json metric: CFR+ iterations/s, beside the CPU path on the same box).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload fhp|leduc_b5|leduc_b3|leduc_pot]
                    [--dump-outputs DIR]

A "step" = one full CFR+ iteration (both seats: value/regret sweep + reach/average sweep each) over the whole public
tree, with the exact best-response evaluation of the current AND the average strategy every `--eval-every` iterations
(inside the timed region).

Default workload `fhp` (BASELINE.json configs[2], the game the metric is quoted on): Flop5Holdem (PokerRL/game/games.py:
222-254) - full game, all C(52,5) = 2 598 960 boards as 134 459 suit-isomorphism classes, 1326-hand ranges, 2 016 890
public nodes, 1 882 430 table rows, run by the board-resident engine (pokerrl_b200/board_engine.py: 17 GB of HBM).  `leduc_b5` (configs[1]) = DiscretizedNLLeduc with
bet_sets.B_5 (873 586 nodes, range 6).  The trees are deterministic: no dataset, no seed.

N > 1 (torchrun): fhp shards the boards over the ranks (strong scaling, one NCCL all-reduce of the chance-node sums per
bottom-up sweep, pokerrl_b200/distributed.py); the Leduc workloads run one independent tree per rank (the reference's
`starting_stack_sizes` axis, weak scaling, no data-path collective).

Rank 0 prints ONE JSON line.  `--impl reference` times the CPU restatement of the reference's path on the host cores
(/root/reference does not exist on the GPU box): the C oracles (OpenMP, all host threads) - oracle/cfr_oracle.c for Leduc;
for fhp, a game the reference cannot run at all (SURVEY.md headline 2), oracle/cfr2_oracle.c (float64, the same O(R)
showdown algorithm class as the GPU) on the first FHP_CPU_BOARDS board classes, a whole fixed instance that the GPU arm
also reports as a matched pair; the full-game figure is that instance scaled by the board count (cost is per board).
"""
import argparse
import contextlib
import io
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

LEDUC = {"leduc_b5": "B_5", "leduc_b3": "B_3", "leduc_pot": "POT_ONLY"}
WORKLOADS = ["fhp", "hulh"] + list(LEDUC) + ["env", "handeval"]
HULH_FLOP = (0, 5, 10)  # 2h 3d 4s


# ---------------------------------------------------------------------------------------------------------- workloads
def make_tree(workload, stack):
    """Leduc workloads: (game class, FlatTree)"""
    from pokerrl_b200.game import bet_sets, games
    from pokerrl_b200.game.flat_tree import FlatTree
    g = games.DiscretizedNLLeduc
    args = g.ARGS_CLS(n_seats=2, starting_stack_sizes_list=[stack, stack],
                      bet_sizes_list_as_frac_of_pot=list(getattr(bet_sets, LEDUC[workload])))
    return g, FlatTree(g, args)


def fhp_args():
    from pokerrl_b200.game import games
    g = games.Flop5Holdem
    return g, g.ARGS_CLS(n_seats=2, starting_stack_sizes_list=[g.DEFAULT_STACK_SIZE] * 2, bet_sizes_list_as_frac_of_pot=[1.0])


def tree_stats(ft):
    import numpy as np
    dec = (ft.kind <= 1) & (ft.first_child >= 0)
    return dict(nodes=int(ft.n_nodes), decision=int(dec.sum()), sum_actions=int(ft.n_slots),
                terminal=int((ft.kind >= 3).sum()), fold=int((ft.kind == 3).sum()), showdown=int((ft.kind == 4).sum()),
                levels=int(ft.n_levels), range=int(ft.R),
                sum_actions_p=[int(ft.n_children[dec & (ft.kind == p)].sum()) for p in (0, 1)],
                decision_p=[int((dec & (ft.kind == p)).sum()) for p in (0, 1)],
                nonterminal=int(((ft.kind <= 2) & (ft.first_child >= 0)).sum()),
                max_level_nodes=int(np.diff(ft.level_start).max()))


def algorithmic_bytes(st, two_card):
    """Minimum bytes ONE seat's two sweeps must move in the level-synchronous design (DESIGN.md §5/§6), rows = range*4 B.
    value sweep: write ev[p] (N rows) + read every child's ev[p] once (N-1) + opponent reach at terminals (T) + regret
                 read/write and strategy read/write at the seat's decision nodes (4 rows per action) + structure
    reach sweep: write reach[p] (N) + read each non-terminal parent row once (NT) + strategy read and average read/write
                 at the seat's nodes (3 rows per action) + structure
    structure = per-node records (16 B record + 4 B work-list entry); two-card trees additionally read the per-board
    strength tables at terminal rows: showdown 3 int16 + 4 uint8 per hand + 2 B x 52 x 51 card rows, fold the card rows.
    Returned seat-averaged: (value_bytes, reach_bytes)."""
    row = st["range"] * 4
    N, T, NT = st["nodes"], st["terminal"], st["nonterminal"]
    sa = sum(st["sum_actions_p"]) / 2.0
    value = row * (N + (N - 1) + T + 4 * sa) + 20 * N
    reach = row * (N + NT + 3 * sa) + 20 * N
    if two_card:
        value += st["showdown"] * (10 * st["range"] + 2 * 52 * 51) + st["fold"] * (2 * 52 * 51)
    return value, reach


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.proc, self.path = None, "/tmp/prl_clocks_%d.csv" % os.getpid()
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=self.f,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        self.proc.wait()
        self.f.close()
        sm, smax, power, reasons = [], None, [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1]))
                smax = float(c[2])
                power.append(float(c[3]))
            except ValueError:
                continue
            for nme, v in zip(names, c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        os.unlink(self.path)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power) if power else None}


# ---------------------------------------------------------------------------------------------------------- CPU arms
def run_cpu_leduc(ft, n_iters, eval_every, threads):
    """C-oracle CFR+ on the host: seconds per iteration (including the evaluation cadence)."""
    import cfr_c
    s = cfr_c.OracleCSolver(ft, "CFRPlus", avg_f64=False, n_threads=threads)
    s.iteration(1)
    t0 = time.perf_counter()
    for i in range(n_iters):
        s.iteration(1)
        if (i + 1) % eval_every == 0:
            s.exploitability_current()
            s.exploitability_average()
    return (time.perf_counter() - t0) / n_iters, s.n_threads


FHP_CPU_BOARDS = 2048  # matched CPU / GPU instance: the first 2048 suit-isomorphism classes


def fhp_subset(spec, n):
    from pokerrl_b200.game.holdem_boards import BoardSpec
    return BoardSpec(spec.boards[:n], spec.board_prob[:n], spec.board_mult[:n], spec.sym_perm, "first %d classes" % n)


def run_cpu_fhp(n_boards, n_iters, threads):
    """oracle/cfr2_oracle.c (float64, OpenMP) CFR+ on the first n_boards classes, lean schedule (what a CFR half-iteration
    needs, i.e. the GPU's schedule).  Returns (seconds per iteration on this instance, threads, exploitability mbb/g)."""
    import numpy as np
    import cfr2_c
    from twocard_common import fhp_tree, oracle_ranks
    from pokerrl_b200.game.games import FlopHoldemRules
    from pokerrl_b200.game.holdem_boards import BoardSpec
    ft = fhp_tree(fhp_subset(BoardSpec.full_game(FlopHoldemRules), n_boards))
    bc = ft.board_cards()
    ranks = np.full((bc.shape[0], ft.R), -1, np.int32)
    ranks[1:] = oracle_ranks(bc[1:])
    c = cfr2_c.Oracle2CSolver(ft, ranks, "CFRPlus", n_threads=threads, lean=True)
    c.iteration(1)
    # thread count: the fastest of {8, 16, 32, 64, all usable} on one iteration each (level-synchronous OpenMP loops stop
    # scaling - and can slow down badly - once the threads outnumber the cores the container really has)
    usable = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else threads
    best = None
    for nt in sorted({min(x, usable) for x in (8, 16, 32, 64, usable)}):
        c.n_threads = c.L.orc2_set_threads(nt)
        t0 = time.perf_counter()
        c.iteration(1)
        dt = time.perf_counter() - t0
        if best is None or dt < best[0]:
            best = (dt, nt)
    c.n_threads = c.L.orc2_set_threads(best[1])
    t0 = time.perf_counter()
    c.iteration(n_iters)
    sec = (time.perf_counter() - t0) / n_iters
    return sec, c.n_threads, c.exploitability_current()


HULH_CPU_CARDS = (1, 8)  # matched CPU / GPU instance of the hulh workload: the first turn card x the first 8 river cards


def hulh_subgame_tree(turn_cards, river_cards):
    """flat tree + constructor arguments of the Limit Hold'em flop sub-game restricted to the first n turn / river cards"""
    from pokerrl_b200.game import games
    from pokerrl_b200.game.flat_tree import FlatTree
    from pokerrl_b200.game.holdem_boards import MultiStreetBoards
    g = games.LimitHoldem
    args = g.ARGS_CLS(n_seats=2, starting_stack_sizes_list=[48, 48], bet_sizes_list_as_frac_of_pot=[1.0])
    free = [c for c in range(52) if c not in HULH_FLOP]
    spec = MultiStreetBoards.subgame(g.RULES, HULH_FLOP, 2, 1, cards_per_layer=[free[:turn_cards], free[:river_cards + turn_cards]])
    return g, args, spec, FlatTree(g, args, board_spec=spec, root_actions=[1, 1])


def run_cpu_hulh(n_iters, threads):
    """oracle/cfr2_oracle.c (float64, OpenMP) Linear CFR on the matched hulh instance: (seconds per iteration, threads,
    river boards of the instance, exploitability mbb/g)"""
    import numpy as np
    import cfr2_c
    from twocard_common import oracle_ranks
    g, args, spec, ft = hulh_subgame_tree(*HULH_CPU_CARDS)
    bc = ft.board_cards()
    ranks = np.full((bc.shape[0], ft.R), -1, np.int32)
    complete = np.nonzero((bc >= 0).sum(axis=1) == 5)[0]
    ranks[complete] = oracle_ranks(bc[complete])
    c = cfr2_c.Oracle2CSolver(ft, ranks, "LinearCFR", n_threads=min(threads, 16), lean=True, ev_normalizer=g.EV_NORMALIZER)
    c.iteration(2)  # first touch of the node arrays
    t0 = time.perf_counter()
    c.iteration(n_iters)
    sec = (time.perf_counter() - t0) / n_iters
    return sec, c.n_threads, int(complete.size), c.exploitability_current()


def run_aux(a):
    """BASELINE.json configs[4]: 2^20 parallel heads-up DiscretizedNLHoldem tables (bet_sets.B_5, stacks 20000, uniformly
    random legal actions from the counter RNG, finished hands re-dealt) and batched 7-card evaluation throughput."""
    import ctypes as C
    import numpy as np
    import torch
    torch.cuda.set_device(0)
    K = a.steps or 200
    W = max(3, a.warmup or 5)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(0)
    time.sleep(0.3)
    if a.workload == "env":
        from pokerrl_b200.game import bet_sets, games
        from pokerrl_b200.game.batched_env import BatchedPokerEnv
        g = games.DiscretizedNLHoldem
        args = g.ARGS_CLS(n_seats=2, starting_stack_sizes_list=[20000, 20000], bet_sizes_list_as_frac_of_pot=bet_sets.B_5)
        B = 1 << 20
        env = BatchedPokerEnv(g, args, B, seed=0)
        env.reset()
        for _ in range(W):
            env.step(None, auto_reset=True)
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(K):
            env.step(None, auto_reset=True)
        ev1.record()
        torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1) / K
        clocks = sampler.stop()
        # e2e: host-provided actions (pinned) in, rewards + done flags out, every step
        acts = torch.zeros(B, dtype=torch.int32).pin_memory()
        rew_h, done_h = torch.zeros(B, 2, dtype=torch.float64).pin_memory(), torch.zeros(B, dtype=torch.uint8).pin_memory()
        acts[:] = 1
        t0 = time.perf_counter()
        for _ in range(20):
            _, r, d, _ = env.step(acts.to("cuda", non_blocking=True), auto_reset=True)
            rew_h.copy_(r, non_blocking=True)
            done_h.copy_(d, non_blocking=True)
            torch.cuda.synchronize()
        e2e = 20 * B / (time.perf_counter() - t0)
        bytes_per_step = B * (4 * 18 * 2 + 52 + env.obs_size * 4 + 16 + 1 + env.N_ACTIONS)
        out = {"metric": "PokerEnv steps/s", "value": B / (ms * 1e-3), "unit": "steps/s", "n_gpus": 1, "steps": K, "warmup": W,
               "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32",
               "data": "synthetic (counter-RNG decks and uniformly random legal actions)",
               "config": {"workload": "2^20 heads-up DiscretizedNLHoldem tables, bet_sets.B_5 (7 actions), stacks 20000, eval "
                                      "mode, random legal play with auto re-deal; obs float32[109] + rewards + done + legal mask "
                                      "written every step"},
               "e2e": {"value": e2e, "unit": "steps/s", "h2d_bytes_per_step": B * 4, "d2h_bytes_per_step": B * 17},
               "gpu_launches": K,
               "roofline": {"bound": "hbm", "kernel": "env_step_kernel", "achieved": bytes_per_step / (ms * 1e-3) / 1e9, "peak": peak,
                            "unit": "GB/s", "frac": bytes_per_step / (ms * 1e-3) / 1e9 / peak, "traffic": None,
                            "algorithmic_bytes_per_launch": bytes_per_step},
               "cpu_baseline": {"value": 18300.0, "unit": "steps/s", "cores": 1, "kind": "reference",
                                "sample": "not re-timed here: the reference env cannot travel to the GPU box; 18.3 k steps/s is "
                                          "the reference's own PokerEnv random play measured in the build container (BASELINE.md)"}}
    else:
        from pokerrl_b200.hand_eval import hand_rank_all_hands_on_given_boards
        rng = np.random.default_rng(0)
        NB = 100000
        boards = torch.from_numpy(np.stack([rng.permutation(52)[:5] for _ in range(NB)]).astype(np.int8)).cuda()
        for _ in range(W):
            out_t = hand_rank_all_hands_on_given_boards(boards)
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(K):
            out_t = hand_rank_all_hands_on_given_boards(boards)
        ev1.record()
        torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1) / K
        clocks = sampler.stop()
        evals = NB * 1081
        import cfr_c  # noqa: F401  (builds oracle/_build)
        orc = C.CDLL(os.path.join(ROOT, "oracle", "_build", "libhand_eval_oracle.so"))
        orc.orc_rank_boards.argtypes = [C.c_void_p, C.c_void_p, C.c_int32]
        hb = np.ascontiguousarray(boards[:4000].cpu().numpy())
        ho = np.zeros((4000, 1326), np.int32)
        t0 = time.perf_counter()
        orc.orc_rank_boards(ho.ctypes.data, hb.ctypes.data, 4000)
        cpu = 4000 * 1081 / (time.perf_counter() - t0)
        assert np.array_equal(ho, out_t[:4000].cpu().numpy())
        b = NB * (5 + 1326 * 4)
        out = {"metric": "7-card hand evaluations/s", "value": evals / (ms * 1e-3), "unit": "evals/s", "n_gpus": 1, "steps": K,
               "warmup": W, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32",
               "data": "synthetic (100 000 random boards, seed 0)",
               "config": {"workload": "100 000 random 5-card boards x 1326 hands (1081 live each), int32 strengths identical to "
                                      "lib_hand_eval.so"},
               "e2e": {"value": None, "unit": "evals/s", "h2d_bytes_per_step": NB * 5, "d2h_bytes_per_step": NB * 1326 * 4},
               "gpu_launches": K,
               "roofline": {"bound": "hbm", "kernel": "rank_boards_kernel", "achieved": b / (ms * 1e-3) / 1e9, "peak": peak,
                            "unit": "GB/s", "frac": b / (ms * 1e-3) / 1e9 / peak, "traffic": None, "algorithmic_bytes_per_launch": b,
                            "note": "integer / LUT-bound, not HBM-bound: ~90 integer instructions per evaluation (rank counting, "
                                    "straight / flush masks) against 5.3 KB written per board; the HBM fraction is reported because "
                                    "the contract asks for one roofline, it is not the limiter"},
               "cpu_baseline": {"value": cpu, "unit": "evals/s", "cores": 1, "kind": "port",
                                "sample": "4 000 boards x 1326 hands by oracle/hand_eval_oracle.c (output compared exactly); the "
                                          "reference binary did 2.73 M evals/s on one core (BASELINE.md)"}}
    out["clocks"] = clocks
    emit((out))


def converge_fhp(a, rank, world, local_rank):
    """BASELINE.json metric, second half: mbb/g exploitability vs wall-clock.  CFR+ on the full game; every --eval-every
    iterations the exact exploitability of the current and of the average strategy is computed (evaluation time is kept
    apart from solve time: both clocks are reported)."""
    import torch
    import torch.distributed as dist
    from pokerrl_b200.board_engine import BoardCFRSolver
    from pokerrl_b200.game.holdem_boards import BoardSpec
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    g, args = fhp_args()
    spec = BoardSpec.full_game(g.RULES)
    if a.fhp_boards:
        spec = fhp_subset(spec, a.fhp_boards)
    s = BoardCFRSolver(g, args, spec, device="cuda:%d" % local_rank, rank=rank, world=world)
    s.iteration(2)
    s.reset()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    curve = [{"iteration": 0, "solve_s": 0.0, "wall_s": 0.0, "mbb_per_g_current": s.exploitability_current(), "mbb_per_g_average": None}]
    solve, t_wall0, it = 0.0, time.perf_counter(), 0
    while it < a.converge:
        n = min(a.eval_every, a.converge - it)
        t0 = time.perf_counter()
        s.iteration(n)
        torch.cuda.synchronize()
        solve += time.perf_counter() - t0
        it += n
        cur, avg = s.exploitability_current(), s.exploitability_average()
        curve.append({"iteration": it, "solve_s": solve, "wall_s": time.perf_counter() - t_wall0, "mbb_per_g_current": cur,
                      "mbb_per_g_average": avg})
    if rank == 0:
        def first_below(x, key):
            for c in curve[1:]:
                if c[key] is not None and c[key] <= x:
                    return {"iteration": c["iteration"], "solve_s": c["solve_s"], "wall_s": c["wall_s"]}
            return None
        emit(({"workload": "Flop5Holdem CFR+ delay 0, %d board classes, range 1326" % spec.boards.shape[0],
                          "n_gpus": world, "iterations": a.converge, "eval_every": a.eval_every,
                          "iterations_per_s_solve_only": a.converge / solve,
                          "time_to_average_strategy_below_mbb_per_g": {str(x): first_below(x, "mbb_per_g_average") for x in (100, 10, 1, 0.1)},
                          "curve": curve}))
    if world > 1:
        dist.destroy_process_group()


def main_fhp(a, rank, world, local_rank):
    """BASELINE.json configs[2] (the game the metric is quoted on): Flop5Holdem CFR+ by the board-resident engine."""
    if a.converge and a.impl != "reference":
        return converge_fhp(a, rank, world, local_rank)
    N_CLASSES = 134459
    K = a.steps if a.steps is not None else 200
    W = max(3, a.warmup if a.warmup is not None else 5)
    nb_used = a.fhp_boards or N_CLASSES
    algo_label = {"CFRPlus": "CFR+", "LinearCFR": "Linear CFR", "VanillaCFR": "Vanilla CFR"}[a.algo]
    cfg = {"workload": "Flop5Holdem %s%s, full game: 134 459 suit-isomorphism classes of the 2 598 960 five-card boards, "
                       "range 1326, stack 20000, exact BR (current+average) every %d iterations%s"
                       % (algo_label, " delay 0" if a.algo == "CFRPlus" else "", a.eval_every,
                          " [DEBUG SUBSET: first %d classes]" % a.fhp_boards if a.fhp_boards else "")}
    ncpu = os.cpu_count() or 1
    if a.impl == "reference" and a.algo != "CFRPlus":
        if rank == 0:
            emit({"impl": "reference", "unavailable": "the CPU arm of the fhp workload times CFR+ (the headline metric)"})
        return
    if a.impl == "reference":
        if rank != 0:
            return
        n_it = max(2, min(K, 8))
        sec, threads, expl = run_cpu_fhp(FHP_CPU_BOARDS, n_it, ncpu)
        v = 1.0 / (sec * nb_used / FHP_CPU_BOARDS)
        sample = ("%d CFR+ iterations of oracle/cfr2_oracle.c (float64, OpenMP, %d threads, the GPU's schedule) on the first %d "
                  "board classes: %.4f s/iteration = %.3f it/s on that instance; scaled by the board count (%d / %d; cost is per "
                  "board) to the full game.  The reference itself cannot run Hold'em trees (SURVEY.md headline 2)"
                  % (n_it, threads, FHP_CPU_BOARDS, sec, 1.0 / sec, nb_used, FHP_CPU_BOARDS))
        emit(({
            "impl": "reference", "metric": "CFR+ iterations/s", "value": v, "unit": "iterations/s", "n_gpus": a.gpus, "steps": n_it,
            "warmup": 1, "ms_per_step": 1e3 / v, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic (deterministic game tree, no dataset)", "config": cfg,
            "matched_instance": {"boards": FHP_CPU_BOARDS, "iterations_per_s": 1.0 / sec, "exploitability_mbb_per_g": expl},
            "cpu_baseline": {"value": v, "unit": "iterations/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    import torch
    import torch.distributed as dist
    from pokerrl_b200 import _native as nat
    from pokerrl_b200.board_engine import BoardCFRSolver
    from pokerrl_b200.game.holdem_boards import BoardSpec

    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # stdout carries exactly one JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = "cuda:%d" % local_rank
    g, args = fhp_args()
    t0 = time.perf_counter()
    spec = BoardSpec.full_game(g.RULES)
    if a.fhp_boards:
        spec = fhp_subset(spec, a.fhp_boards)
    t_spec = time.perf_counter() - t0
    t0 = time.perf_counter()
    s = BoardCFRSolver(g, args, spec, algo=a.algo, device=dev, rank=rank, world=world)
    torch.cuda.synchronize()
    t_setup = time.perf_counter() - t0
    L = s.L
    collective = s.collective

    def steps(solver, i0, n):
        out, i = [], i0
        while i < i0 + n:
            m = min(a.eval_every - (i % a.eval_every), i0 + n - i)
            solver.iteration(m)
            i += m
            if i % a.eval_every == 0:
                out.append((i, solver.exploitability_current(), solver.exploitability_average()))
        return out

    steps(s, 0, W)
    s.reset()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler is not None:
        time.sleep(0.5)
    steps(s, 0, W)
    s.reset()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    launches0, n_ar0 = nat.lib().prl_launch_count(), s.n_allreduce
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    wall0 = time.perf_counter()
    ev0.record()
    trace = steps(s, 0, K)
    ev1.record()
    torch.cuda.synchronize()
    wall = time.perf_counter() - wall0
    dev_ms = ev0.elapsed_time(ev1)
    launches = nat.lib().prl_launch_count() - launches0
    n_allreduce = s.n_allreduce - n_ar0
    clocks = sampler.stop() if sampler else None
    t = torch.tensor([dev_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.barrier()
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    max_ms = float(t.item())
    if a.dump_outputs and rank == 0:  # before the roofline launches below change the tables
        dump_outputs(a.dump_outputs, board_engine_outputs(s, trace))

    # --- roofline of the dominant kernel (board_sweep_kernel, update form), CUDA events on its stream around each launch
    def ev_pair():
        return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    sw, half, evals = [], [], []
    for rep in range(5):
        for p in (0, 1):
            e0, e1 = ev_pair()
            e0.record()
            s._pending[1 - p] = 1.0 if a.algo != "CFRPlus" else 0.0  # Vanilla / Linear: the sweep also adds the opponent's average
            s._sweep_begin(s.bufs, p, False, 0, 0)
            e1.record()
            torch.cuda.synchronize()
            sw.append(e0.elapsed_time(e1))
    for rep in range(4):  # whole half-iterations (sweep + cross-rank sum + trunk chain)
        for p in (0, 1):
            e0, e1 = ev_pair()
            e0.record()
            s._update_begin(p)
            s._update_end(p)
            e1.record()
            torch.cuda.synchronize()
            half.append(e0.elapsed_time(e1))
        s.iter_counter += 1
    for rep in range(2):
        e0, e1 = ev_pair()
        e0.record()
        s.exploitability_current()
        s.exploitability_average()
        e1.record()
        torch.cuda.synchronize()
        evals.append(e0.elapsed_time(e1))
    sweep_ms, half_ms, eval_ms = statistics.median(sw), statistics.median(half), statistics.median(evals)
    rows_bytes = L["ldb"] * 4
    # algorithmic bytes of ONE update launch (DESIGN.md §6): per board 7 opponent regret rows read, 7 own regret rows read +
    # written, 7 own average rows read + written (35 rows of 1088 floats) + the board's 15 392-byte index tables, once
    per_board = 35 * rows_bytes + L["blob"]
    bytes_launch = s.n_boards * per_board
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = bytes_launch / (sweep_ms * 1e-3) / 1e9
    traffic, traffic_note = None, "no ncu capture recorded under profiles/"
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "r02_fhp_sweep_traffic.json")))
        traffic = tr["dram_bytes_per_board"] * s.n_boards
        traffic_note = tr["note"]
    except Exception:
        pass
    it_ms = max_ms / K
    # SURVEY.md §8(d): B_min = 16 R sum(A) + 4 R n_boards per iteration with R = 1326 (regret + average read and written once)
    b_min = (16 * 1326 * 14 + 4 * 1326) * (N_CLASSES if not a.fhp_boards else a.fhp_boards)
    roofline = {
        "bound": "hbm", "kernel": "board_sweep_kernel<ShapeFHP, seat, update> (persistent, 2 CTAs per SM, one (board, seat) unit at a "
                                  "time; 2 launches per iteration = %.0f %% of the iteration)" % (100 * 2 * sweep_ms / (2 * half_ms)),
        "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
        "peak_source": "MEASURED_PEAKS.json" if "hbm_gbs" in peaks else "fallback 6.65 TB/s",
        "algorithmic_bytes_per_launch": bytes_launch, "launch_ms": sweep_ms, "traffic": traffic, "traffic_note": traffic_note,
        "bytes_per_board": {"rows": 35 * rows_bytes, "index_tables": L["blob"]},
        "frac_vs_Bmin": {"B_min_bytes_per_iteration": b_min * (1.0 / world if world > 1 else 1.0),
                         "achieved_GBps": b_min / world / (2 * half_ms * 1e-3) / 1e9,
                         "frac": b_min / world / (2 * half_ms * 1e-3) / 1e9 / peak,
                         "note": "SURVEY.md §8(d) minimum with R = 1326 over a plain iteration (2 half-iterations, no BR pass)"},
        "time_shares_ms": {"update_sweep_per_seat": sweep_ms, "half_iteration": half_ms,
                           "trunk_and_cross_rank_sum_per_half_iteration": half_ms - sweep_ms,
                           "exploitability_current_plus_average": eval_ms, "timed_step_avg": it_ms},
    }

    # --- matched CPU / GPU instance + shard-invariance proof (small engines on this rank's GPU)
    matched = None
    if rank == 0:
        small = BoardCFRSolver(g, args, fhp_subset(BoardSpec.full_game(g.RULES), FHP_CPU_BOARDS), device=dev)
        small.iteration(3)
        torch.cuda.synchronize()
        e0, e1 = ev_pair()
        e0.record()
        small.iteration(20)
        e1.record()
        torch.cuda.synchronize()
        matched = {"boards": FHP_CPU_BOARDS, "gpu_iterations_per_s": 20e3 / e0.elapsed_time(e1)}
        del small
    invariance = None
    if world > 1:
        sub = fhp_subset(BoardSpec.full_game(g.RULES), 1024)
        part = BoardCFRSolver(g, args, sub, device=dev, rank=rank, world=world)
        part.iteration(5)
        mine = [part.exploitability_current(), part.exploitability_average()]
        chk = part.bufs.regret.double().sum().item()
        if rank == 0:
            one = BoardCFRSolver(g, args, sub, device=dev)
            one.iteration(5)
            ref = [one.exploitability_current(), one.exploitability_average()]
            invariance = {"boards": 1024, "iterations": 5, "sharded": mine, "single_rank_replay": ref,
                          "max_abs_diff": max(abs(x - y) for x, y in zip(mine, ref)),
                          "trunk_regret_checksum_equal": chk == one.bufs.regret.double().sum().item()}
            del one
        del part

    # --- e2e: the user-facing call (CFRPlus facade: iteration() + logging through ChiefBase, results read on the host)
    import importlib
    CFRPlus = getattr(importlib.import_module("pokerrl_b200.cfr." + a.algo), a.algo)  # CFRPlus / LinearCFR / VanillaCFR facade
    from pokerrl_b200.game import games
    from pokerrl_b200.rl.base_cls.workers.ChiefBase import ChiefBase
    del s
    torch.cuda.empty_cache()
    chief = ChiefBase(t_prof=None)
    with contextlib.redirect_stdout(io.StringIO()):
        kw = dict(delay=0) if a.algo == "CFRPlus" else {}
        cfr = CFRPlus(name="bench", chief_handle=chief, game_cls=games.Flop5Holdem, agent_bet_set=[1.0],
                      eval_every=a.eval_every, device=dev, board_spec=spec, **kw)
    for _ in range(W):
        cfr.iteration()
    cfr.reset()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0t = time.perf_counter()
    for _ in range(K):
        cfr.iteration()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - e0t
    t2 = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
    e2e_s = float(t2.item())
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    out = {
        "metric": algo_label + " iterations/s", "value": K / (max_ms * 1e-3), "unit": "iterations/s", "n_gpus": world, "steps": K,
        "warmup": W, "ms_per_step": it_ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic (deterministic game tree, no dataset)",
        "config": dict(cfg, boards_per_rank=s_n_boards(nb_used, rank, world), engine="board-resident (pokerrl_b200/board_engine.py)",
                       l2="per-rank tables %.1f GB >> 126 MB L2 (no explicit flush)" % (
                           2 * s_n_boards(nb_used, rank, world) * 14 * rows_bytes / 2 ** 30),
                       parallelism="boards round-robin over %d ranks; per bottom-up sweep ONE cross-rank sum of the chance node's "
                                   "int64 fixed-point vector (%d in the timed region): %s" % (world, n_allreduce, collective)),
        "clocks": clocks,
        "e2e": {"value": K / e2e_s, "unit": "iterations/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 2 * 8 * (K // a.eval_every) / K,
                "note": "CFRPlus.iteration() facade incl. ChiefBase logging; CFR has no per-step host input - the one-off setup "
                        "(board enumeration, hand ranks + index tables built on the GPU) is reported under setup"},
        "setup": {"board_spec_s": t_spec, "engine_build_s": t_setup, "note": "outside every timed number"},
        "gpu_launches": int(launches), "wall_ms_per_step": wall * 1e3 / K,
        "exploitability_trace_mbb_per_g": trace[-3:], "roofline": roofline, "matched_instance": matched,
    }
    if invariance is not None:
        out["shard_invariance"] = invariance
    if world == 1 and not a.no_cpu_baseline and a.algo == "CFRPlus":
        n_it = 6
        sec, threads, expl = run_cpu_fhp(FHP_CPU_BOARDS, n_it, ncpu)
        out["matched_instance"].update(cpu_iterations_per_s=1.0 / sec, cpu_threads=threads, same_config=True,
                                       ratio=out["matched_instance"]["gpu_iterations_per_s"] * sec)
        out["cpu_baseline"] = {"value": 1.0 / (sec * nb_used / FHP_CPU_BOARDS), "unit": "iterations/s", "cores": threads, "kind": "port",
                               "sample": "%d CFR+ iterations of oracle/cfr2_oracle.c (float64, OpenMP, %d threads) on the first %d board "
                                         "classes at %.4f s/iteration, scaled by the board count to the full game (cost is per board); "
                                         "the reference cannot run Hold'em trees at all (SURVEY.md headline 2)"
                                         % (n_it, threads, FHP_CPU_BOARDS, sec)}
    emit((out))
    if world > 1:
        dist.destroy_process_group()


def s_n_boards(n, rank, world):
    return len(range(rank, n, world))


DUMP_LIMIT_BYTES = 64 << 20
DUMP_BOARDS = 256  # 256 boards x 2 tables x 14 rows x 1088 floats = 30.5 MB


def board_engine_outputs(s, trace):
    """What a caller of the timed fhp path receives - BoardCFRSolver.state_dict() and the exploitability trace - with the
    per-board tables cut to the rows of a fixed, seeded sample of DUMP_BOARDS of this rank's boards, each board's rows in the
    order of the post-deal tree's nodes: [boards, rows per board, ldb]."""
    import numpy as np
    import torch
    s.flush_average()
    rng = np.random.default_rng(0)
    boards = np.sort(rng.choice(s.n_boards, min(DUMP_BOARDS, s.n_boards), replace=False))
    own_rows = [r0 for _, (r0, _) in sorted(s.local_rows.items())]
    rows = torch.from_numpy((boards[:, None] * s.rows_per_board + np.array(own_rows)[None, :]).reshape(-1)).to(s.regret.device)
    shape = (boards.size, len(own_rows), s.regret.shape[1])
    return {"exploitability": np.array(trace, np.float64).reshape(-1, 3),  # (iteration, current, average) in mbb/g
            "regret_rows": s.regret[rows].cpu().numpy().reshape(shape), "avg_rows": s.avg[rows].cpu().numpy().reshape(shape),
            "trunk_regret": s.bufs.regret.cpu().numpy(), "trunk_strat": s.bufs.strat.cpu().numpy(),
            "trunk_avg": s.bufs.avg.cpu().numpy()}


def dump_outputs(out_dir, arrays):
    """out_dir/<name>.npy for every array (float32 / float64 only, at most DUMP_LIMIT_BYTES in all)"""
    import numpy as np
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise ValueError("outputs of %d bytes exceed the %d-byte dump limit" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if a.dtype not in (np.float32, np.float64):
            raise TypeError("%s: dtype %s is neither float32 nor float64" % (name, a.dtype))
        np.save(os.path.join(out_dir, name + ".npy"), a)


_REAL_STDOUT = None


def emit(obj):
    """the ONE JSON line of this process on the real stdout (fd 1 is pointed at stderr while the benchmark runs, so that
    banners of NCCL / the launcher cannot end up in front of it)"""
    sys.stdout.flush()
    if _REAL_STDOUT is not None:
        os.dup2(_REAL_STDOUT, 1)
    print(json.dumps(obj))
    sys.stdout.flush()


def main():
    global _REAL_STDOUT
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="fhp", choices=WORKLOADS)
    ap.add_argument("--eval-every", type=int, default=20)
    ap.add_argument("--algo", default="CFRPlus", choices=["CFRPlus", "LinearCFR", "VanillaCFR"],
                    help="fhp workload: the algorithm the board engine runs (the headline metric is CFRPlus)")
    ap.add_argument("--fhp-boards", type=int, default=0, help="debug: only the first n isomorphism classes")
    ap.add_argument("--hulh-turns", type=int, default=0, help="hulh: only the first n turn cards (memory: the full 49 need >= 2 GPUs)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--converge", type=int, default=0, metavar="ITERS",
                    help="fhp / hulh: run ITERS iterations and print the exploitability-vs-wall-clock curve (one JSON line) "
                         "instead of the throughput line; evaluation every --eval-every iterations")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="fhp: after the timed steps write what they computed as DIR/<name>.npy (float32 / float64, <= 64 MB: "
                         "exploitability trace, trunk tables, the table rows of a fixed seeded sample of %d boards)" % DUMP_BOARDS)
    a = ap.parse_args()
    if a.steps is not None and a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.workload != "fhp" or a.impl != "b200" or a.converge):
        ap.error("--dump-outputs covers the timed GPU run of the fhp workload")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if a.workload in ("env", "handeval"):
        if rank == 0 and a.impl == "b200":
            run_aux(a)
        elif rank == 0:
            emit(({"impl": "reference", "unavailable": "aux workloads carry their CPU baseline in the main line"}))
        return
    if a.workload == "fhp":
        return main_fhp(a, rank, world, local_rank)
    hulh = a.workload == "hulh"
    fhp = a.workload in ("fhp", "hulh")  # the hulh sub-game runs on the level engine (two chance layers)
    algo_name = "LinearCFR" if hulh else "CFRPlus"
    K = a.steps if a.steps is not None else (40 if fhp else 2000)
    W = max(3, a.warmup if a.warmup is not None else (3 if fhp else 20))
    N_CLASSES = 134459
    if hulh:
        cfg = {"workload": "LimitHoldem (blinds 1/2, bets 2/4, 4 raises per round, stack 48) Linear CFR on the public sub-game "
                           "rooted at the flop 2h3d4s after SB limps / BB checks: turn (49 cards) and river (48 cards) chance "
                           "layers, 190 954 round-subtrees, range 1326, exact BR (current+average) every %d iterations%s"
                           % (a.eval_every, " [DEBUG: first %d turn cards]" % a.hulh_turns if a.hulh_turns else "")}
    elif fhp:
        cfg = {"workload": "Flop5Holdem CFR+ delay 0, full game: 134 459 suit-isomorphism classes of the 2 598 960 "
                           "five-card boards, range 1326, stack 20000, exact BR (current+average) every %d iterations"
                           % a.eval_every}
    else:
        cfg = {"workload": "DiscretizedNLLeduc CFR+ delay 0, bet_sets.%s, stack 20000%s, exact BR (current+average) "
                           "every %d iterations" % (LEDUC[a.workload], " + 1000*rank (one tree per rank)" if world > 1 else "",
                                                    a.eval_every)}

    # ------------------------------------------------------------------ reference arm (CPU restatement)
    if a.impl == "reference":
        if rank != 0:
            return
        ncpu = os.cpu_count() or 1
        if hulh:
            emit(({"impl": "reference", "unavailable": "no CPU arm for the hulh sub-game workload (the float64 oracle is "
                              "exercised on a restricted sub-game in tests/test_gpu_twocard.py)"}))
            return
        if True:
            g, ft = make_tree(a.workload, 20000)
            K = min(K, 200)
            sec, threads = run_cpu_leduc(ft, K, a.eval_every, min(ncpu, 16))
            cfg.update(tree=tree_stats(ft))
            v, ms = 1.0 / sec, sec * 1e3
            sample = "%d full CFR+ iterations of the same tree by oracle/cfr_oracle.c (OpenMP)" % K
        emit(({
            "impl": "reference", "metric": "CFR+ iterations/s", "value": v, "unit": "iterations/s", "n_gpus": a.gpus,
            "steps": K, "warmup": 1, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong" if fhp else "weak", "vs_baseline": None, "dtype": "f64" if fhp else "f32",
            "data": "synthetic (deterministic game tree, no dataset)", "config": cfg,
            "cpu_baseline": {"value": v, "unit": "iterations/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }))
        return

    # ------------------------------------------------------------------ B200 arm
    import torch
    import torch.distributed as dist
    from pokerrl_b200 import _native as nat
    from pokerrl_b200.solver import CFRSolver

    torch.cuda.set_device(local_rank)
    if world > 1:
        # stdout carries exactly one JSON line: NCCL's own banner / debug output (NCCL_DEBUG set on the box) goes to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = "cuda:%d" % local_rank
    t0 = time.perf_counter()
    spec = None
    if fhp:
        from pokerrl_b200.distributed import ShardedCFRSolver
        from pokerrl_b200.game.holdem_boards import BoardSpec
        root_actions = None
        if hulh:
            from pokerrl_b200.game import games
            from pokerrl_b200.game.holdem_boards import MultiStreetBoards
            g = games.LimitHoldem
            args = g.ARGS_CLS(n_seats=2, starting_stack_sizes_list=[48, 48], bet_sizes_list_as_frac_of_pot=[1.0])
            free = [c for c in range(52) if c not in HULH_FLOP]
            cpl = [free[:a.hulh_turns], free] if a.hulh_turns else None
            spec = MultiStreetBoards.subgame(g.RULES, HULH_FLOP, 2, 1, cards_per_layer=cpl)
            root_actions = [1, 1]
        else:
            g, args = fhp_args()
            spec = BoardSpec.full_game(g.RULES)
        if a.fhp_boards and not hulh:
            spec = BoardSpec(spec.boards[:a.fhp_boards], spec.board_prob[:a.fhp_boards], spec.board_mult[:a.fhp_boards],
                             spec.sym_perm, "first %d classes (debug)" % a.fhp_boards)
            cfg["workload"] += " [DEBUG SUBSET: %d classes]" % a.fhp_boards
        t_build = time.perf_counter() - t0
        t0 = time.perf_counter()
        s = ShardedCFRSolver(g, args, spec, algo_name, device=dev, rank=rank, world=world, root_actions=root_actions)
        ft = s.ft
    else:
        g, ft = make_tree(a.workload, 20000 + 1000 * rank)
        t_build = time.perf_counter() - t0
        t0 = time.perf_counter()
        s = CFRSolver(ft, "CFRPlus", delay=0, avg_f64=False, device=dev)
    torch.cuda.synchronize()
    t_upload = time.perf_counter() - t0
    st = tree_stats(ft)
    tree_bytes = sum(t.numel() * t.element_size() for k, t in vars(s.dtree).items()
                     if k.startswith("t_") and isinstance(t, torch.Tensor))

    def steps(i0, n):
        """n steps starting at step index i0; iterations between two evaluations share one call"""
        out, i = [], i0
        while i < i0 + n:
            m = min(a.eval_every - (i % a.eval_every), i0 + n - i)
            s.iteration(m)
            i += m
            if i % a.eval_every == 0:
                out.append((i, s.exploitability_current(), s.exploitability_average()))
        return out

    steps(0, W)
    s.reset()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler is not None:
        time.sleep(0.5)  # let nvidia-smi start sampling while the GPU runs untimed steps
    steps(0, W)
    s.reset()
    torch.cuda.synchronize()

    # --- timed region: K steps, device-timed with CUDA events on the launching stream, barrier + sync on both sides
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    launches0 = nat.lib().prl_launch_count()
    n_ar0 = getattr(s, "n_allreduce", 0)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    wall0 = time.perf_counter()
    ev0.record()
    trace = steps(0, K)
    ev1.record()
    torch.cuda.synchronize()
    wall = time.perf_counter() - wall0
    dev_ms = ev0.elapsed_time(ev1)
    launches = nat.lib().prl_launch_count() - launches0
    clocks = sampler.stop() if sampler else None
    t = torch.tensor([dev_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.barrier()
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    max_ms = float(t.item())
    n_allreduce = getattr(s, "n_allreduce", 0) - n_ar0

    # --- roofline of the dominant kernels, timed live with CUDA events on their stream (sweep by sweep, after the run)
    import ctypes as C
    from pokerrl_b200.solver import _stream
    vb, rb = algorithmic_bytes(st, fhp)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    psrc = "MEASURED_PEAKS.json" if "hbm_gbs" in peaks else "fallback 6.65 TB/s"
    if fhp:
        tree_p, buf_p = C.byref(s.dtree.desc), C.byref(s.bufs.desc)
        v_ms, r_ms = [], []
        for rep in range(4):
            for p in (0, 1):
                e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
                e[0].record()
                s._value_sweep(s.bufs, 1 << p, False, s.algo, p, s.modes)
                e[1].record()
                nat.call("prl_reach_update", tree_p, buf_p, s.algo, p, s.iter_counter, s.delay, _stream())
                e[2].record()
                torch.cuda.synchronize()
                if rep >= 1:
                    v_ms.append(e[0].elapsed_time(e[1]))
                    r_ms.append(e[1].elapsed_time(e[2]))
            s.iter_counter += 1
        vm, rm = statistics.mean(v_ms), statistics.mean(r_ms)
        achieved = vb / (vm * 1e-3) / 1e9
        roofline = {"bound": "hbm", "kernel": "value/regret sweep of one seat = fold2_kernel + terminal2_kernel_v3 + value2_kernel_v2<false,true> + "
                    "chance_*_kernel over all %d levels (terminal2_kernel is the largest share, see profiles/)" % st["levels"],
                    "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": psrc,
                    "algorithmic_bytes_per_sweep": vb, "sweep_ms": vm, "traffic": None,
                    "traffic_note": "no full-game ncu --set full capture (110 GB resident; replay save/restore); the 20 000-"
                    "board capture in profiles/r01_g_twocard_v2.md has terminal2_kernel at 25.1 KB DRAM per terminal row "
                    "(10.6 KB of rows + the board's tables, shared by neighbouring rows through L2) and reach2_kernel_v2 "
                    "at 22.9 KB per node on the widest level (3 rows in, 2 rows out = 26.5 KB algorithmic; part of a "
                    "20 000-board level still sits in L2)",
                    "reach_sweep": {"kernel": "reach2_kernel_v2<true> x %d levels" % st["levels"], "algorithmic_bytes": rb,
                                    "sweep_ms": rm, "achieved": rb / (rm * 1e-3) / 1e9, "frac": rb / (rm * 1e-3) / 1e9 / peak}}
    else:
        it_ms = []
        for rep in range(12):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            s.iteration(a.eval_every)
            e1.record()
            torch.cuda.synchronize()
            if rep >= 2:
                it_ms.append(e0.elapsed_time(e1))
        l_ms = statistics.mean(it_ms)
        bpl = a.eval_every * 2 * (vb + rb)
        achieved = bpl / (l_ms * 1e-3) / 1e9
        kname = ("cfr_iterations_kernel<6,2> (persistent cooperative kernel: %d CFR+ iterations = %d level steps with grid "
                 "barriers per launch)" % (a.eval_every, a.eval_every * 2 * (2 * st["levels"] - 1)))
        roofline = {"bound": "hbm", "kernel": kname,
                    "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": psrc,
                    "algorithmic_bytes_per_launch": bpl, "launch_ms": l_ms, "traffic": None,
                    "note": "latency/occupancy-bound, not HBM-bound: R = 6 rows, 27 dependent level steps per seat"}

    # --- e2e: the user-facing call (CFRPlus façade: iteration() + logging through ChiefBase, results read on the host)
    from pokerrl_b200.cfr.CFRPlus import CFRPlus
    from pokerrl_b200.game import bet_sets, games
    from pokerrl_b200.rl.base_cls.workers.ChiefBase import ChiefBase
    del s
    torch.cuda.empty_cache()
    chief = ChiefBase(t_prof=None)
    with contextlib.redirect_stdout(io.StringIO()):
        if hulh:
            cfr = None  # the facade constructs full games; the sub-game is driven through the engine API (same calls)
        elif fhp:
            cfr = CFRPlus(name="bench", chief_handle=chief, game_cls=games.Flop5Holdem, agent_bet_set=[1.0], delay=0,
                          eval_every=a.eval_every, device=dev, board_spec=spec)
        else:
            cfr = CFRPlus(name="bench", chief_handle=chief, game_cls=games.DiscretizedNLLeduc,
                          agent_bet_set=list(getattr(bet_sets, LEDUC[a.workload])),
                          starting_stack_sizes=[20000 + 1000 * rank], delay=0, eval_every=a.eval_every, device=dev)
    if cfr is None:
        s = ShardedCFRSolver(g, args, spec, algo_name, device=dev, rank=rank, world=world, root_actions=root_actions)

        class _Engine:  # iteration + host read-back of the exploitability numbers at the evaluation cadence
            n = 0

            def iteration(self):
                s.iteration(1)
                self.n += 1
                if self.n % a.eval_every == 0:
                    return s.exploitability_current(), s.exploitability_average()

            def reset(self):
                s.reset()
                self.n = 0
        cfr = _Engine()
    for _ in range(W):
        cfr.iteration()
    cfr.reset()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0 = time.perf_counter()
    for _ in range(K):
        cfr.iteration()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - e0
    t2 = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
    e2e_s = float(t2.item())
    d2h_per_step = 2 * 8 * (K // a.eval_every) / K  # two float32[2] exploitability read-backs per evaluation

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    jobs = 1 if fhp else world  # fhp: ONE game sharded over the ranks; Leduc: one tree per rank
    out = {
        "metric": ("Linear CFR" if hulh else "CFR+") + " iterations/s", "value": jobs * K / (max_ms * 1e-3), "unit": "iterations/s", "n_gpus": world,
        "steps": K, "warmup": W, "ms_per_step": max_ms / K, "higher_is_better": True,
        "scaling": "strong" if fhp else "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic (deterministic game tree, no dataset)",
        "config": dict(cfg, tree_per_rank=st,
                       l2="per-rank working set %.1f GB >> 126 MB L2 (no explicit flush)" % (
                           (6 * st["nodes"] + 3 * st["sum_actions"]) * st["range"] * 4 / 2 ** 30),
                       parallelism=("boards sharded over %d ranks, one NCCL all-reduce of the chance-node sums per bottom-up "
                                    "sweep (%d in the timed region)" % (world, n_allreduce)) if fhp
                       else "one tree per rank (stack-size axis), no collective"),
        "clocks": clocks,
        "e2e": {"value": jobs * K / e2e_s, "unit": "iterations/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": d2h_per_step,
                "note": "CFRPlus.iteration() facade incl. ChiefBase logging; CFR has no per-step host input - the one-off "
                        "tree / board-table upload is reported under setup"},
        "setup": {"tree_build_s": t_build, "upload_and_tables_s": t_upload, "tree_h2d_bytes": int(tree_bytes)},
        "gpu_launches": int(launches),
        "wall_ms_per_step": wall * 1e3 / K,
        "exploitability_trace_mbb_per_g": trace[-3:],
        "roofline": roofline,
    }
    if world == 1 and not a.no_cpu_baseline:
        ncpu = os.cpu_count() or 1
        if hulh:
            # matched instance (first turn card x 8 river cards) on both sides; the CPU figure scaled by the river-board count
            g2, args2, spec2, _ = hulh_subgame_tree(*HULH_CPU_CARDS)
            small = ShardedCFRSolver(g2, args2, spec2, "LinearCFR", device=dev, root_actions=[1, 1])
            small.iteration(3)
            torch.cuda.synchronize()
            e0m, e1m = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0m.record()
            small.iteration(20)
            e1m.record()
            torch.cuda.synchronize()
            gpu_its = 20e3 / e0m.elapsed_time(e1m)
            sec, threads, n_river_small, _ = run_cpu_hulh(4, ncpu)
            n_river = int(sum(1 for _ in range(len(spec.boards[2]))))
            out["matched_instance"] = {"turn_x_river_cards": list(HULH_CPU_CARDS), "river_boards": n_river_small,
                                       "gpu_iterations_per_s": gpu_its, "cpu_iterations_per_s": 1.0 / sec, "cpu_threads": threads,
                                       "same_config": True, "ratio": gpu_its * sec}
            out["cpu_baseline"] = {"value": 1.0 / (sec * n_river / n_river_small), "unit": "iterations/s", "cores": threads,
                                   "kind": "port",
                                   "sample": "4 Linear-CFR iterations of oracle/cfr2_oracle.c (float64, OpenMP, %d threads) on the "
                                             "sub-game restricted to %d turn x %d river cards (%d river boards) at %.4f s/iteration, "
                                             "scaled by the river-board count (%d here) - the cost is dominated by the river rounds; "
                                             "the reference cannot run Hold'em trees at all (SURVEY.md headline 2)"
                                             % (threads, HULH_CPU_CARDS[0], HULH_CPU_CARDS[1], n_river_small, sec, n_river)}
        else:
            n = max(2, min(K, int(15.0 / max(0.014 * st["nodes"] / 873586.0, 1e-4))))
            n = (n // a.eval_every) * a.eval_every or n
            sec, threads = run_cpu_leduc(ft, n, a.eval_every, min(ncpu, 16))
            out["cpu_baseline"] = {"value": 1.0 / sec, "unit": "iterations/s", "cores": threads, "kind": "port",
                                   "sample": "%d full CFR+ iterations (same tree, same BR cadence) by oracle/cfr_oracle.c "
                                             "with OpenMP; the reference's own Python path is ~400x slower per node "
                                             "(BASELINE.md: 0.448 s/iter on the 1 096-node tree)" % n}
    emit((out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
