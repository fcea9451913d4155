"""Arguments of the head-to-head evaluator (`PokerRL/eval/head_to_head/H2HArgs.py`): hands per seat, plus where and how the
matches run - the device, the seed of the deals and decisions, and the number of tables played in lockstep per batch."""


class H2HArgs:
    def __init__(self, n_hands, device=None, seed=0, batch_size=1 << 20):
        self.n_hands = n_hands
        self.device = device
        self.seed = seed
        self.batch_size = batch_size
