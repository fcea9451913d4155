"""drop-in namespace: PokerRL.eval.head_to_head"""
