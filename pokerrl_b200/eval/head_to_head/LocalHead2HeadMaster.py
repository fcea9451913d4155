"""Head-to-head evaluator master (`PokerRL/eval/head_to_head/LocalHead2HeadMaster.py:10-126`): two modes of an eval agent
play `n_hands` hands per seat against each other; agent 0's mean winnings are logged with their 95 % confidence interval
under the reference's experiment names ("<name> <mode>_stack_<s>: Head2Head_Winnings Total / Conf_lower95 / Conf_upper95",
several stacks: "<name> Head2HeadMulti_Stack: Head2Head_Winnings Averaged Total").  The matches run through `play_match`:
on the device when both agents expose `device_policy()`, otherwise the reference's per-hand loop.  Stacks at which an
agent cannot compute its mode are skipped and left out of the multi-stack average."""
from pokerrl_b200.eval._.EvaluatorMasterBase import EvaluatorMasterBase
from pokerrl_b200.eval.head_to_head.match import play_match
from pokerrl_b200.rl.base_cls.TrainingProfileBase import get_env_builder

_MULTI_STACK_MODE = "Head2Head"


class LocalHead2HeadMaster(EvaluatorMasterBase):
    def __init__(self, t_prof, chief_handle, eval_agent_cls):
        super().__init__(t_prof=t_prof, eval_env_bldr=get_env_builder(t_prof), chief_handle=chief_handle,
                         eval_type="Head2Head_Winnings", log_conf_interval=True)
        self._args = t_prof.module_args["h2h"]
        self._env_bldr = get_env_builder(t_prof)
        assert self._env_bldr.N_SEATS == 2
        self._eval_agents = [eval_agent_cls(t_prof=t_prof) for _ in range(self._env_bldr.N_SEATS)]
        self._REFERENCE_AGENT = 0
        if self._is_multi_stack and _MULTI_STACK_MODE not in self._exp_name_multi_stack:
            new, et = chief_handle.create_experiment, "Head2Head_Winnings"
            self._exp_name_multi_stack[_MULTI_STACK_MODE] = new("%s %sMulti_Stack: %s Averaged Total" % (t_prof.name, _MULTI_STACK_MODE, et))
            self._exp_names_multi_stack_conf[_MULTI_STACK_MODE] = [new("%s %s: %s Conf_%s" % (t_prof.name, _MULTI_STACK_MODE, et, b))
                                                                  for b in ("lower95", "upper95")]

    def set_modes(self, modes):
        for e, mode in zip(self._eval_agents, modes):
            e.set_mode(mode)

    def update_weights(self):
        w = self.pull_current_strat_from_chief()
        for e in self._eval_agents:
            e.update_weights(w)

    def evaluate(self, iter_nr):
        means, halves = [], []
        for stack_size_idx, stack_size in enumerate(self._t_prof.eval_stack_sizes):
            for e in self._eval_agents:
                e.set_stack_size(stack_size=stack_size)
            if not all(e.can_compute_mode() for e in self._eval_agents):
                continue
            mean, d = self._run_eval(stack_size)
            self._log_results(iter_nr=iter_nr, agent_mode=self._eval_agents[self._REFERENCE_AGENT].get_mode(),
                              stack_size_idx=stack_size_idx, score=mean, upper_conf95=mean + d, lower_conf95=mean - d)
            means.append(mean)
            halves.append(d)
        if self._is_multi_stack and means:
            m, d = sum(means) / len(means), sum(halves) / len(halves)
            self._log_multi_stack(agent_mode=_MULTI_STACK_MODE, iter_nr=iter_nr, score_total=m, lower_conf95=m - d,
                                  upper_conf95=m + d)

    def _run_eval(self, stack_size):
        a = self._args
        return play_match(self._eval_agents[self._REFERENCE_AGENT], self._eval_agents[1 - self._REFERENCE_AGENT], a.n_hands,
                          stack_size, seed=a.seed, batch_size=a.batch_size, device=a.device)
