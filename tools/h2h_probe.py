"""Head-to-head throughput on one GPU: one JSON line per game with hands/s of the device path (2^20 tables in lockstep) and
of the per-hand host loop (a few thousand hands), kernel-inclusive match time from CUDA events, and the card's name and power
limit read in the same run.

    python tools/h2h_probe.py [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def agents(game, bet_set, iters):
    from pokerrl_b200.cfr.CFRPlus import CFRPlus
    from pokerrl_b200.cfr.TabularCFREvalAgent import TabularCFREvalAgent
    from pokerrl_b200.rl.base_cls.TrainingProfileBase import TrainingProfileBase
    from pokerrl_b200.rl.base_cls.workers.ChiefBase import ChiefBase
    cfr = CFRPlus(name="p", chief_handle=ChiefBase(None), game_cls=game, agent_bet_set=list(bet_set), delay=0)
    for _ in range(iters):
        cfr.iteration()
    t_prof = TrainingProfileBase("p", game, list(bet_set))
    a = TabularCFREvalAgent.from_cfr(t_prof, cfr)
    del cfr
    torch.cuda.empty_cache()
    ft, fp = a.own_tree()
    inv = 1.0 / ft.n_children[ft.parent[np.nonzero(ft.slot >= 0)[0]]].astype(np.float32)
    b = TabularCFREvalAgent(t_prof=t_prof)
    if isinstance(a._table, torch.Tensor):
        b.update_weights((torch.from_numpy(inv).cuda()[:, None].expand(-1, a._table.shape[1]).contiguous(), fp))
    else:
        b.update_weights((np.repeat(inv[:, None], ft.R, axis=1), fp))
    return a, b


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--host-hands", type=int, default=1000, help="hands per seat of the host loop")
    args = ap.parse_args()
    from pokerrl_b200.eval.head_to_head.match import play_match_details
    from pokerrl_b200.game import bet_sets, games
    lines = []
    for name, bet_set, iters in (("StandardLeduc", bet_sets.POT_ONLY, 100), ("DiscretizedNLLeduc", bet_sets.B_3, 100),
                                 ("Flop5Holdem", [1.0], 3)):
        game = getattr(games, name)
        a, b = agents(game, bet_set, iters)
        stack = [game.DEFAULT_STACK_SIZE] * 2
        n = 1 << 19  # per seat: 2^20 tables in one batch
        play_match_details(a, b, n, stack, seed=1)  # warm-up (tree upload, deal map, module load)
        times = []
        for rep in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            d = play_match_details(a, b, n, stack, seed=2 + rep)
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1) / 1e3)
        t = time.perf_counter()
        h = play_match_details(a, b, args.host_hands, stack, host_loop=True)
        t_host = time.perf_counter() - t
        line = {"game": name, "card": card(), "device_tables": 2 * n, "device_match_s": min(times),
                "device_hands_per_s": 2 * n / min(times), "device_mean_mbb": d["mean"], "device_half_width_mbb": d["half_width"],
                "host_hands": h["n"], "host_s": t_host, "host_hands_per_s": h["n"] / t_host}
        print(json.dumps(line), flush=True)
        lines.append(line)
        del a, b
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()
