"""PPOKL_Agent.train restated on the CPU: the executable definition the device PPOKL_Agent is tested against.

The reference's ppokl_agent.py cannot run as written (DESIGN.md §8 f3): it reads `policy.representation_actor` (:22), builds
the Atari buffer for every env (:26), and calls `learner.update` with six arguments and `aux_batch['old_logp']` (:80-82)
against the five-argument `PPOKL_Learner.update`.  Corrected, the file is PPOCLIP_Agent's loop with the
`{"old_dist": None}` auxiliary and `PPOKL_Learner.update(obs, act, ret, adv, old_dists)`.  So this port is oracle.ref_port.PPOAgentPort's loop (pinned to
the live reference agent) with OldDistBufferPort storing the old distributions and `ppokl_update` (pinned to the
reference's goldens) carrying `{"kl_coef"}` from update to update; the action and permutation tapes are PPOAgentPort's.
"""
import numpy as np
import torch

from oracle import ref_port


class PPOKLAgentPort(ref_port.PPOAgentPort):
    """`record=True` keeps the actions and permutations drawn, for a device agent to replay; `kl_trace` lists, per update,
    (the minibatch's KL, the coefficient that update used, the coefficient after it)."""

    def __init__(self, envs, policy, optimizer, scheduler, n_steps, n_epoch, n_minibatch, gamma, gae_lam, vf_coef=0.25,
                 ent_coef=0.01, target_kl=0.001, use_gae=True, use_advnorm=True, use_obsnorm=False, use_rewnorm=False,
                 obsnorm_range=5, rewnorm_range=5, action_tape=None, perm_tape=None, record=False, kl_coef=1.0):
        act_shape = () if not hasattr(envs.action_space, "low") else envs.action_space.shape
        memory = ref_port.OldDistBufferPort(envs.observation_space.shape, act_shape, envs.num_envs, n_steps, use_gae,
                                            use_advnorm, gamma, gae_lam)
        super().__init__(envs, policy, optimizer, scheduler, n_steps, n_epoch, n_minibatch, gamma, gae_lam, use_gae=use_gae,
                         use_advnorm=use_advnorm, use_obsnorm=use_obsnorm, use_rewnorm=use_rewnorm,
                         obsnorm_range=obsnorm_range, rewnorm_range=rewnorm_range, memory=memory, action_tape=action_tape,
                         perm_tape=perm_tape)
        self.kl_hp = dict(vf_coef=vf_coef, ent_coef=ent_coef, target_kl=target_kl)
        self.kl_state = {"kl_coef": float(kl_coef)}
        self.kl_trace = []
        self.recorded_actions, self.recorded_perms = ([], []) if record else (None, None)

    def _act(self, obs, taped):
        _, dist, v = self.policy(obs)
        a = dist.stochastic_sample() if taped is None else torch.as_tensor(taped, device=v.device)
        if self.recorded_actions is not None:
            self.recorded_actions.append(a.detach().cpu().numpy().copy())
        return a.detach().cpu().numpy(), v.detach().cpu().numpy(), dist

    def _shuffle(self, indexes):
        super()._shuffle(indexes)
        if self.recorded_perms is not None:
            self.recorded_perms.append(indexes.copy())

    def update(self, obs, act, ret, adv, old):
        used = self.kl_state["kl_coef"]
        info = ref_port.ppokl_update(self.policy, self.optimizer, self.scheduler, (obs, act, ret, adv), old, self.kl_state,
                                     **self.kl_hp)
        self.kl_trace.append((info["kl"], used, self.kl_state["kl_coef"]))
        return info

    def train(self, train_steps):
        # a copy: without the observation normaliser the reference's first stored observation aliases the env's buffer,
        # which the step overwrites; the device agent stores the observation the action was computed from
        obs = self.envs.buf_obs.copy()
        mem = self.memory
        for _ in range(train_steps):
            self.obs_rms.update(obs)
            obs = self._obs(obs)
            taped = None
            if self.action_tape is not None:
                taped = self.action_tape[self._tape_pos]
                self._tape_pos += 1
            acts, value, dists = self._act(obs, taped)
            next_obs, rewards, terminals, truncations, infos = self.envs.step(acts)
            mem.store(obs, acts, self._rew(rewards), value, terminals, {"old_dist": dists})
            if mem.full:
                vals = self.policy(self._obs(next_obs))[2].detach().cpu().numpy()
                for i in range(self.n_envs):
                    mem.finish_path(0.0 if terminals[i] else vals[i], i)
                indexes = np.arange(self.buffer_size)
                for _ in range(self.n_epoch):
                    self._shuffle(indexes)
                    for start in range(0, self.buffer_size, self.batch_size):
                        o, a, r, _, ad, aux = mem.sample(indexes[start:start + self.batch_size])
                        self.last_info = self.update(o, a, r, ad, aux["old_dist"])
                mem.clear()
            self.returns = (1 - terminals) * self.gamma * self.returns + rewards
            obs = next_obs
            for i in range(self.n_envs):
                if terminals[i] or truncations[i]:
                    self.ret_rms.update(self.returns[i:i + 1])
                    self.returns[i] = 0.0
                    if terminals[i]:
                        mem.finish_path(0.0, i)
                    else:
                        mem.finish_path(self.policy(self._obs(next_obs))[2].detach().cpu().numpy()[i], i)
                    obs[i] = infos[i]["reset_obs"]
                    self.episodes += 1
            self.current_step += self.n_envs
