"""ctypes binding of libpokerrl_b200.so (the C ABI declared in include/pokerrl_b200.h).

There is NO CPU fallback: if the library is missing or a call fails this module raises.  The numpy/C oracle under
oracle/ is test infrastructure and is never imported from here.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# PRL_LIB_PATH: another build of the same library (tools/build_variants.py writes kernel-variant builds for A/B timing)
LIB_PATH = os.environ.get("PRL_LIB_PATH") or os.path.join(_HERE, "lib", "libpokerrl_b200.so")

# enums of include/pokerrl_b200.h
KIND_P0, KIND_P1, KIND_CHANCE, KIND_FOLD, KIND_SHOWDOWN, KIND_SHOWDOWN_ALLIN = range(6)
ALGO_VANILLA, ALGO_CFR_PLUS, ALGO_LINEAR = 0, 1, 2
ABI_VERSION = 4  # include/pokerrl_b200.h: PRL_ABI_VERSION
STRAT_F32, STRAT_UNIFORM64, STRAT_AVG_F64, STRAT_AVG_SUM, STRAT_AVG_F32 = range(5)


class PrlTree(C.Structure):
    _fields_ = [
        ("n_nodes", C.c_int32), ("n_levels", C.c_int32), ("n_slots", C.c_int32), ("n_range", C.c_int32),
        ("ld", C.c_int32), ("n_hole", C.c_int32), ("n_deck", C.c_int32), ("n_suits", C.c_int32),
        ("pair_bonus", C.c_int32), ("max_actions", C.c_int32),
        ("level_start", C.c_void_p),
        ("parent", C.c_void_p), ("first_child", C.c_void_p), ("n_children", C.c_void_p), ("slot", C.c_void_p),
        ("kind", C.c_void_p), ("acted_last", C.c_void_p), ("pot", C.c_void_p), ("board", C.c_void_p),
        ("order", C.c_void_p), ("level_nonterm", C.c_void_p), ("meta", C.c_void_p),
        ("level_ndec", C.c_void_p), ("hand_cards", C.c_void_p), ("n_boards", C.c_int32),
        ("max_chance_children", C.c_int32), ("board_mask", C.c_void_p), ("board_prob", C.c_void_p),
        ("board_mult", C.c_void_p), ("board_gs", C.c_void_p), ("board_ge", C.c_void_p), ("board_pos", C.c_void_p),
        ("board_row_order", C.c_void_p), ("board_row_pos", C.c_void_p), ("board_complete", C.c_void_p),
        ("n_sym", C.c_int32), ("sym_perm", C.c_void_p), ("eq_const", C.c_float), ("board_hand_rec", C.c_void_p),
        ("node_rec2", C.c_void_p), ("work_rec2", C.c_void_p), ("level_nfold", C.c_void_p),
        ("level_nallin", C.c_void_p), ("allin_nodes", C.c_void_p), ("allin_pot", C.c_void_p), ("allin_tiles", C.c_void_p),
        ("allin_partial", C.c_void_p),
    ]


class PrlBuffers(C.Structure):
    _fields_ = [("reach", C.c_void_p), ("ev", C.c_void_p), ("ev_br", C.c_void_p), ("regret", C.c_void_p),
                ("strat", C.c_void_p), ("avg", C.c_void_p), ("workspace", C.c_void_p),
                ("workspace_bytes", C.c_uint64)]


class PrlBoardGame(C.Structure):
    _fields_ = [("n_boards", C.c_int32), ("n_range", C.c_int32), ("ld", C.c_int32), ("n_deck", C.c_int32),
                ("n_local", C.c_int32), ("frac_bits", C.c_int32), ("grid", C.c_int32), ("eq_const", C.c_float),
                ("kind", C.c_int8 * 16), ("parent", C.c_int8 * 16), ("first_child", C.c_int8 * 16),
                ("n_children", C.c_int8 * 16), ("acted_last", C.c_int8 * 16), ("pot", C.c_float * 16),
                ("row0", C.c_int64 * 16), ("row_m", C.c_int32 * 16),
                ("tables", C.c_void_p), ("board_prob", C.c_void_p), ("board_mult", C.c_void_p), ("regret", C.c_void_p),
                ("avg", C.c_void_p), ("w_private", C.c_void_p), ("w_total", C.c_void_p)]


class PrlTrunk(C.Structure):
    _fields_ = [("n_nodes", C.c_int32), ("chance_node", C.c_int32), ("n_buf_nodes", C.c_int32), ("ld", C.c_int32),
                ("n_range", C.c_int32), ("mode", C.c_int32 * 2), ("eq_const", C.c_float),
                ("kind", C.c_int8 * 8), ("first_child", C.c_int8 * 8), ("n_children", C.c_int8 * 8), ("acted_last", C.c_int8 * 8),
                ("first_slot", C.c_int32 * 8), ("pot", C.c_float * 8), ("hand_cards", C.c_void_p), ("reach", C.c_void_p),
                ("ev", C.c_void_p), ("ev_br", C.c_void_p), ("regret", C.c_void_p), ("strat", C.c_void_p), ("avg", C.c_void_p)]


class PrlEnvCfg(C.Structure):
    _fields_ = [
        ("n_envs", C.c_int32), ("kind", C.c_int32), ("n_actions", C.c_int32), ("n_rounds", C.c_int32),
        ("n_round_slots", C.c_int32), ("n_hole", C.c_int32), ("n_ranks", C.c_int32), ("n_suits", C.c_int32),
        ("n_deck", C.c_int32), ("n_flop", C.c_int32), ("n_turn", C.c_int32), ("n_river", C.c_int32),
        ("small_blind", C.c_int32), ("big_blind", C.c_int32), ("ante", C.c_int32), ("small_bet", C.c_int32),
        ("big_bet", C.c_int32), ("round_big_bet_starts", C.c_int32), ("max_raises", C.c_int32 * 4),
        ("first_action_no_call", C.c_int32), ("limit_raise_is_pot", C.c_int32), ("btn_first_postflop", C.c_int32),
        ("suits_matter", C.c_int32), ("pair_bonus", C.c_int32), ("start_stack", C.c_int32 * 2), ("obs_size", C.c_int32),
        ("fracs", C.c_double * 32), ("reward_scalar", C.c_double), ("norm", C.c_double),
    ]


class PrlH2H(C.Structure):
    _fields_ = [("n_envs", C.c_int32), ("n_range", C.c_int32), ("n_hole", C.c_int32), ("chance_by_class", C.c_int32),
                ("max_decisions", C.c_int32), ("seat_swap_at", C.c_int64), ("hand0", C.c_int64), ("seed", C.c_uint64),
                ("kind", C.c_void_p), ("first_child", C.c_void_p), ("n_children", C.c_void_p), ("first_slot", C.c_void_p),
                ("action", C.c_void_p), ("table_a", C.c_void_p), ("table_b", C.c_void_p), ("ld_a", C.c_int64),
                ("ld_b", C.c_int64), ("board_class", C.c_void_p), ("board_perm", C.c_void_p), ("sym_perm", C.c_void_p),
                ("uniforms", C.c_void_p), ("node", C.c_void_p), ("n_dec", C.c_void_p), ("perm", C.c_void_p),
                ("chips", C.c_void_p), ("desync", C.c_void_p)]


_lib = None


def lib():
    """Loads the CUDA library on first use; raises if it has not been built (python -m pokerrl_b200.csrc.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "pokerrl_b200: CUDA library %s is missing. Build it with `python -m pokerrl_b200.csrc.build` "
            "(or __graft_entry__.build()). There is no CPU fallback." % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    L.prl_abi_version.restype = C.c_int
    if L.prl_abi_version() != ABI_VERSION:
        raise RuntimeError("pokerrl_b200: %s was built for ABI %d, the Python side expects %d - rebuild it with "
                           "`python -m pokerrl_b200.csrc.build`" % (LIB_PATH, L.prl_abi_version(), ABI_VERSION))
    L.prl_last_error.restype = C.c_char_p
    tp, bp, ip = C.POINTER(PrlTree), C.POINTER(PrlBuffers), C.POINTER(C.c_int)
    L.prl_reach_pass.argtypes = [tp, bp, C.c_int, ip, C.c_void_p]
    L.prl_value_pass.argtypes = [tp, bp, C.c_int, C.c_int, ip, C.c_void_p]
    L.prl_root_exploitability.argtypes = [tp, bp, C.c_void_p, C.c_void_p]
    L.prl_cfr_half_iteration.argtypes = [tp, bp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, ip, C.c_void_p]
    L.prl_cfr_sweep.argtypes = [tp, bp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, ip, C.c_int, C.c_void_p]
    L.prl_launch_count.restype = C.c_ulonglong
    L.prl_cfr_iterations.argtypes = [tp, bp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, ip, C.c_void_p]
    L.prl_evaluate.argtypes = [tp, bp, ip, C.c_int, C.c_void_p, C.c_void_p]
    L.prl_pack_node_meta.argtypes = [tp, C.c_void_p, C.c_void_p]
    for f in ("prl_reach_pass", "prl_value_pass", "prl_root_exploitability", "prl_cfr_half_iteration", "prl_cfr_sweep", "prl_pack_node_meta", "prl_cfr_iterations",
              "prl_evaluate"):
        getattr(L, f).restype = C.c_int
    L.prl_value_levels.argtypes = [tp, bp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, ip, C.c_int, C.c_int,
                                   C.c_int, C.c_void_p]
    L.prl_reach_update.argtypes = [tp, bp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
    L.prl_value_levels.restype = L.prl_reach_update.restype = C.c_int
    L.prl_reach_levels.argtypes = [tp, bp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, ip, C.c_int, C.c_int, C.c_void_p]
    L.prl_reach_levels.restype = C.c_int
    L.prl_board_order_tables.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_void_p, C.c_void_p]
    L.prl_board_order_tables.restype = C.c_int
    L.prl_hand_rank_boards.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    L.prl_hand_rank_7.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    for f in ("prl_hand_rank_boards", "prl_hand_rank_7"):
        getattr(L, f).restype = C.c_int
    L.prl_gather_agent_policy.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                          C.c_void_p]
    L.prl_gather_agent_policy.restype = C.c_int
    L.prl_lbr_workspace_doubles.argtypes = [C.c_int, C.c_int]
    L.prl_lbr_workspace_doubles.restype = C.c_longlong
    L.prl_lbr_checkdown_equity.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                           C.c_void_p]
    L.prl_lbr_checkdown_equity.restype = C.c_int
    L.prl_allin_tiles_bytes.argtypes = L.prl_allin_partial_bytes.argtypes = [C.c_int]
    L.prl_allin_tiles_bytes.restype = L.prl_allin_partial_bytes.restype = C.c_int64
    L.prl_allin_equity_accumulate.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    L.prl_allin_equity_finish.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    L.prl_allin_values.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                   C.c_void_p]
    for f in ("prl_allin_equity_accumulate", "prl_allin_equity_finish", "prl_allin_values"):
        getattr(L, f).restype = C.c_int
    gp = C.POINTER(PrlBoardGame)
    L.prl_board_layout.argtypes = [C.POINTER(C.c_int32)]
    L.prl_board_grid.argtypes = []
    L.prl_board_rows.argtypes = [C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
    L.prl_board_rows.restype = C.c_int
    L.prl_board_shape_ok.argtypes = [gp]
    L.prl_board_build_tables.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    L.prl_board_sweep.argtypes = [gp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int,
                                  C.c_void_p]
    L.prl_board_collect.argtypes = [gp, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]
    L.prl_board_permute.argtypes = [gp, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                    C.c_void_p]
    L.prl_board_trunk.argtypes = [gp, C.POINTER(PrlTrunk), C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                  C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_int, C.c_void_p]
    L.prl_board_trunk.restype = C.c_int
    for f in ("prl_board_layout", "prl_board_grid", "prl_board_shape_ok", "prl_board_build_tables", "prl_board_sweep",
              "prl_board_collect", "prl_board_permute"):
        getattr(L, f).restype = C.c_int
    ep = C.POINTER(PrlEnvCfg)
    L.prl_env_state_fields.restype = C.c_int
    L.prl_env_reset.argtypes = [ep, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_int,
                                C.c_void_p]
    L.prl_env_step.argtypes = [ep, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                               C.c_uint64, C.c_uint64, C.c_int, C.c_void_p]
    L.prl_env_reset.restype = L.prl_env_step.restype = C.c_int
    hp = C.POINTER(PrlH2H)
    L.prl_h2h_init.argtypes = [hp, C.c_void_p, C.c_void_p]
    L.prl_h2h_step.argtypes = [hp, ep, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.prl_h2h_collect.argtypes = [hp, C.c_double, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]
    L.prl_h2h_init.restype = L.prl_h2h_step.restype = L.prl_h2h_collect.restype = C.c_int
    _lib = L
    return L


def call(name, *args):
    """Calls an entry point and raises RuntimeError(prl_last_error()) on a non-zero status."""
    L = lib()
    rc = getattr(L, name)(*args)
    if rc != 0:
        raise RuntimeError("%s failed (%d): %s" % (name, rc, L.prl_last_error().decode()))


def modes(m0, m1):
    return (C.c_int * 2)(m0, m1)
