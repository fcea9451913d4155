from pokerrl_b200.eval.head_to_head.H2HArgs import H2HArgs  # noqa: F401
from pokerrl_b200.eval.head_to_head.LocalHead2HeadMaster import LocalHead2HeadMaster  # noqa: F401
from pokerrl_b200.eval.head_to_head.match import exact_head_to_head, play_match  # noqa: F401
