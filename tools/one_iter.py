"""Profiling helper: a few persistent CFR+ iterations on the B_5 Leduc tree (used under ncu)."""
import os, sys
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bench import make_tree
from pokerrl_b200.solver import CFRSolver
g, ft = make_tree(sys.argv[1] if len(sys.argv) > 1 else "leduc_b5", 20000)
s = CFRSolver(ft, "CFRPlus")
for _ in range(4):
    s.iteration(1)
torch.cuda.synchronize()
print(s.exploitability_current())
