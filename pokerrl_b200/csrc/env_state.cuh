// Layout of the batched env's table state (csrc/env_kernels.cu): SoA int32[kFields][n_envs], one field per row.
// Shared with the kernels that read a table's state between env steps (csrc/h2h.cu).
#pragma once

namespace prl_env {
enum Field {
    F_ROUND, F_POT, F_STACK0, F_STACK1, F_BET0, F_BET1, F_FLAGS, F_CUR, F_LAST_RAISER, F_N_ACT_EP, F_N_RAISES,
    F_CAPPED, F_CAP_RAISER, F_CAP_NOREOPEN, F_LAST_TYPE, F_LAST_AMT, F_LAST_WHO, F_DONE, kFields
};
}  // namespace prl_env
