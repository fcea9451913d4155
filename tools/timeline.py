import os, sys, ctypes as C, torch, numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bench import make_tree
from pokerrl_b200 import _native as nat
from pokerrl_b200.solver import CFRSolver
g, ft = make_tree("leduc_b5", 20000)
s = CFRSolver(ft, "CFRPlus")
s.iteration(5)
buf = torch.zeros(4096, dtype=torch.int64, device="cuda")
nat.lib().prl_debug_set_timeline(C.c_void_p(buf.data_ptr()))
s.iteration(2)
torch.cuda.synchronize()
nat.lib().prl_debug_set_timeline(None)
t = buf.cpu().numpy()
L = ft.n_levels
n = 1 + 2 * 2 * (L + L - 1)
d = np.diff(t[:n]) / 1e3
per_iter = 2 * (L + L - 1)
it = d[per_iter:2 * per_iter]
print("levels", L, "iteration total us", it.sum())
print("value p0:", np.round(it[:L], 1))
print("reach p0:", np.round(it[L:2 * L - 1], 1))
print("value p1:", np.round(it[2 * L - 1:3 * L - 1], 1))
print("reach p1:", np.round(it[3 * L - 1:], 1))
print("level sizes (deep->top):", np.diff(ft.level_start)[::-1])
