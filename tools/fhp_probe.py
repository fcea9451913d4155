"""Probe: full Flop5Holdem (134 459 isomorphism classes) on one GPU - build time, memory, iteration time."""
import os, sys, time
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pokerrl_b200.game import games
from pokerrl_b200.game.flat_tree import FlatTree
from pokerrl_b200.game.holdem_boards import BoardSpec
from pokerrl_b200.solver import CFRSolver
g = games.Flop5Holdem
args = g.ARGS_CLS(n_seats=2, starting_stack_sizes_list=[20000] * 2, bet_sizes_list_as_frac_of_pot=[1.0])
t = time.time(); spec = BoardSpec.full_game(g.RULES); print("boards", spec.note, "%.1fs" % (time.time() - t), flush=True)
nb = int(sys.argv[1]) if len(sys.argv) > 1 else spec.boards.shape[0]
if nb < spec.boards.shape[0]:
    spec = BoardSpec(spec.boards[:nb], spec.board_prob[:nb], spec.board_mult[:nb], spec.sym_perm, "first %d classes" % nb)
t = time.time(); ft = FlatTree(g, args, board_spec=spec); print("tree", ft.n_nodes, ft.n_slots, "%.1fs" % (time.time() - t), flush=True)
t = time.time(); s = CFRSolver(ft, "CFRPlus"); torch.cuda.synchronize(); print("upload+tables %.1fs" % (time.time() - t), "mem GB", torch.cuda.memory_allocated() / 2**30, flush=True)
for i in range(3):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); s.iteration(1); e1.record(); torch.cuda.synchronize()
    print("iteration ms", e0.elapsed_time(e1), flush=True)
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record(); c = s.exploitability_current(); e1.record(); torch.cuda.synchronize(); print("eval current ms", e0.elapsed_time(e1), c, flush=True)
e0.record(); a = s.exploitability_average(); e1.record(); torch.cuda.synchronize(); print("eval average ms", e0.elapsed_time(e1), a, "mem GB", torch.cuda.max_memory_allocated() / 2**30, flush=True)
