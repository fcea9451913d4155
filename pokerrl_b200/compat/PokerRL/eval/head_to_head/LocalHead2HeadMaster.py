from pokerrl_b200.eval.head_to_head.LocalHead2HeadMaster import LocalHead2HeadMaster  # noqa: F401
