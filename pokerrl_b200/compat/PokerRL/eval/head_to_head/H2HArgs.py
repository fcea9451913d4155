from pokerrl_b200.eval.head_to_head.H2HArgs import H2HArgs  # noqa: F401
