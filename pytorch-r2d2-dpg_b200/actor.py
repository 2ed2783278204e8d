"""Drop-in for the reference's actor.py: `Actor(actor_id)`, `.run()`, `.load_model()`,
`.calc_nstep_reward()`, `.calc_priorities()`, `actor_process(actor_id)` (actor.py:16-180).

The actor is OUTSIDE the accelerated hot path (SURVEY 8: CPU actors stay as they are); this module
exists so the reference's r2d2.py imports and runs unchanged, and it keeps the episode tuple, recurrent
state and memory{i}.pt formats the learner ingests.  Without dm_control it steps a synthetic
environment of the configured shape (BASELINE.json configs[4]: "Humanoid-shape synthetic env").

With R2D2_ACTOR_ENVS=n, actor_process runs VecActor instead: n environments in lockstep, the four nets stepped on a
GPU in one batched call per vector step (r2d2_b200.acting.ActEngine).  Unset, it is the CPU Actor below.
"""
import os
from collections import deque
from copy import deepcopy
from time import sleep

import numpy as np
import torch

from models import ActorNet, CriticNet
from replay_memory import ReplayMemory
from utils import calc_priority, get_obs, invertical_vf


class _SyntheticEnv:
    """Random linear dynamics with the dm_control TimeStep surface (reset/step/last/observation/reward)."""

    class _TS:
        def __init__(self, obs, reward, last):
            self.observation, self.reward, self._last = {"o": obs}, reward, last

        def last(self):
            return self._last

    def __init__(self, obs_size, n_actions, episode_len=250, seed=0):
        self.rng = np.random.default_rng(seed)
        self.obs_size, self.n_actions, self.episode_len = obs_size, n_actions, episode_len
        self.A = self.rng.standard_normal((obs_size, obs_size)).astype(np.float32) * 0.1
        self.Bm = self.rng.standard_normal((n_actions, obs_size)).astype(np.float32) * 0.5

    def action_spec(self):
        return type("Spec", (), {"shape": (self.n_actions,)})()

    def reset(self):
        self.t = 0
        self.x = self.rng.standard_normal(self.obs_size).astype(np.float32)
        return self._TS(self.x, 0.0, False)

    def step(self, action):
        self.t += 1
        self.x = np.tanh(self.x @ self.A + np.asarray(action, np.float32) @ self.Bm).astype(np.float32)
        return self._TS(self.x, float(-np.square(self.x).mean()), self.t >= self.episode_len * 4)


def _make_env(actor_id):
    if "R2D2_OBS_SIZE" not in os.environ:
        try:
            from dm_control import suite
            return suite.load(domain_name="walker", task_name="run")
        except ImportError:
            pass
    return _SyntheticEnv(int(os.environ.get("R2D2_OBS_SIZE", 24)), int(os.environ.get("R2D2_N_ACTIONS", 6)),
                         seed=actor_id)


def actor_process(actor_id):
    n_envs = os.environ.get("R2D2_ACTOR_ENVS")
    actor = VecActor(actor_id, int(n_envs)) if n_envs else Actor(actor_id)
    actor.run()


class Actor:
    def __init__(self, actor_id):
        self.env = _make_env(actor_id)
        self.action_size = self.env.action_spec().shape[0]
        self.obs_size = get_obs(self.env.reset().observation).shape[1]
        self.actor_id = actor_id
        self.burn_in_length, self.learning_length, self.n_step = 20, 40, 5
        self.sequence_length = self.burn_in_length + self.learning_length
        self.sequence, self.recurrent_state, self.priority = [], [], []
        self.td_loss = deque(maxlen=self.learning_length)
        self.memory_sequence_size = 1000
        self.memory = ReplayMemory(memory_sequence_size=self.memory_sequence_size)
        self.memory_save_interval = 3
        self.gamma = 0.997
        self.actor_parameter_update_interval = 500
        self.model_path = './model_data/'
        self.hidden = int(os.environ.get("R2D2_HIDDEN", 128))
        self.device = torch.device(os.environ.get("R2D2_ACTOR_DEVICE", "cpu"))  # actors are CPU workers here
        self.actor = ActorNet(self.obs_size, self.action_size, 0, hidden=self.hidden).to(self.device).eval()
        self.target_actor = deepcopy(self.actor)
        self.critic = CriticNet(self.obs_size, self.action_size, 0, hidden=self.hidden).to(self.device).eval()
        self.target_critic = deepcopy(self.critic)
        self.load_model()

    def _nets(self):
        return (("actor", self.actor), ("target_actor", self.target_actor), ("critic", self.critic),
                ("target_critic", self.target_critic))

    def load_model(self):
        """Follow the learner's model.pt (actor.py:50-72); retried while the file is being replaced."""
        path = self.model_path + 'model.pt'
        if not os.path.isfile(path):
            return
        for _ in range(20):
            try:
                model_dict = torch.load(path, map_location=self.device)
                for name, net in self._nets():
                    net.load_state_dict(model_dict[name])
                return
            except Exception:
                sleep(np.random.rand() * 2 + 0.5)

    def calc_nstep_reward(self):
        """Overwrite rewards with their n-step discounted sums (actor.py:74-76)."""
        for i in range(len(self.sequence) - self.n_step):
            self.sequence[i][2][0] = sum(self.sequence[i + j][2][0] * (self.gamma ** j) for j in range(self.n_step))

    @torch.no_grad()
    def calc_priorities(self):
        """Initial sequence priorities by replaying the episode through the four nets (actor.py:78-107)."""
        for _, net in self._nets():
            net.reset_state()
        self.td_loss = deque(maxlen=self.learning_length)
        self.priority = []
        t = lambda a: torch.from_numpy(np.asarray(a, np.float32)).to(self.device).unsqueeze(0)  # noqa: E731
        for i in range(self.n_step):
            nxt = t(self.sequence[i][0])
            self.target_critic(nxt, self.target_actor(nxt))
        for i in range(len(self.sequence) - self.n_step):
            obs, action, nxt = t(self.sequence[i][0]), t(self.sequence[i][1]), t(self.sequence[i + self.n_step][0])
            q = self.critic(obs, action).cpu().numpy()
            q_next = self.target_critic(nxt, self.target_actor(nxt)).cpu().numpy()
            if i >= self.burn_in_length:
                terminal = self.sequence[i + self.n_step - 1][3][0]
                y = self.sequence[i][2][0] + (self.gamma ** self.n_step) * (1.0 - terminal) * q_next
                y = invertical_vf(torch.tensor(y)).numpy()
                self.td_loss.append((q - y).mean())
            if i >= self.sequence_length:
                self.priority.append(calc_priority(np.array(list(self.td_loss), dtype=np.float32) ** 2.0))

    def run(self, max_episodes=None):
        episode = step = 0
        while max_episodes is None or episode < max_episodes:
            time_step = self.env.reset()
            obs = get_obs(time_step.observation)
            for _, net in self._nets():
                net.reset_state()
            self.sequence, self.recurrent_state, self.priority = [], [], []
            episode += 1
            reward_sum = 0.0
            while not time_step.last():
                states = [net.get_state() for _, net in self._nets()]
                with torch.no_grad():
                    x = torch.from_numpy(obs).to(self.device)
                    action = self.actor(x)
                    self.critic(x, action)
                    self.target_critic(x, self.target_actor(x))
                action = np.clip(action.cpu().numpy()[0] + np.random.normal(0, 0.3, self.action_size), -1, 1)
                reward = 0.0
                for _ in range(4):                                        # action repeat, actor.py:152-157
                    time_step = self.env.step(action)
                    next_obs = get_obs(time_step.observation)
                    reward += time_step.reward or 0.0
                    if time_step.last():
                        break
                reward_sum += reward
                step += 1
                self.sequence.append((obs[0], action.astype(np.float32), [reward], [1.0 if time_step.last() else 0.0]))
                self.recurrent_state.append([[h[0], c[0]] for h, c in states])
                obs = next_obs.copy()
                if step % self.actor_parameter_update_interval == 0:
                    self.load_model()
            if self.actor_id == 0:
                print('episode:', episode, 'step:', step, 'reward:', reward_sum)
            if len(self.sequence) >= self.sequence_length:
                pad = (np.zeros(self.obs_size, np.float32), np.zeros(self.action_size, np.float32), [0.0], [1.0])
                self.sequence.extend([(pad[0].copy(), pad[1].copy(), [0.0], [1.0]) for _ in range(self.n_step)])
                self.calc_nstep_reward()
                self.calc_priorities()
                self.memory.add(self.sequence, self.recurrent_state, self.priority)
            if len(self.memory.memory) > self.memory_save_interval:
                self.memory.save(self.actor_id)


class VecActor:
    """`n_envs` environments stepped in lockstep with the four nets on the GPU (r2d2_b200.acting.ActEngine: one
    batched step per vector step instead of four batch-1 calls per environment).  Selected by actor_process when
    R2D2_ACTOR_ENVS is set; writes the same episode tuples, recurrent states and memory{i}.pt files as Actor.

    Env k gets seed actor_id * n_envs + k, and the exploration noise is one np.random.normal(0, 0.3, (n_envs, A)) draw
    per vector step, so n_envs = 1 reproduces Actor's seeds and noise sequence.  Episodes that finish in the same step
    get their n-step rewards and initial priorities from ONE batched r2d2_b200.actor_priority.episode_priorities call.
    Device: R2D2_ACTOR_DEVICE if it names a CUDA device, else cuda:0."""

    def __init__(self, actor_id, n_envs):
        from r2d2_b200.acting import ActEngine
        if n_envs < 1:
            raise ValueError("n_envs >= 1")
        self.actor_id, self.n_envs = actor_id, n_envs
        self.envs = [_make_env(actor_id * n_envs + k) for k in range(n_envs)]
        self.action_size = self.envs[0].action_spec().shape[0]
        self.obs_size = get_obs(self.envs[0].reset().observation).shape[1]
        self.burn_in_length, self.learning_length, self.n_step = 20, 40, 5
        self.sequence_length = self.burn_in_length + self.learning_length
        self.memory_sequence_size = 1000
        self.memory = ReplayMemory(memory_sequence_size=self.memory_sequence_size)
        self.memory_save_interval = 3
        self.gamma = 0.997
        self.actor_parameter_update_interval = 500
        self.model_path = './model_data/'
        self.hidden = int(os.environ.get("R2D2_HIDDEN", 128))
        dev = os.environ.get("R2D2_ACTOR_DEVICE", "")
        self.device = torch.device(dev if dev.startswith("cuda") else "cuda:0")
        # the same freshly initialised nets as Actor (same torch RNG draws) until model.pt exists
        actor = ActorNet(self.obs_size, self.action_size, 0, hidden=self.hidden)
        critic = CriticNet(self.obs_size, self.action_size, 0, hidden=self.hidden)
        self.weights = {"actor": actor.state_dict(), "target_actor": deepcopy(actor.state_dict()),
                        "critic": critic.state_dict(), "target_critic": deepcopy(critic.state_dict())}
        self.engine = ActEngine(self.obs_size, self.action_size, self.hidden, n_envs, self.device)
        self.engine.load(self.weights)
        self.load_model()

    def load_model(self):
        """Follow the learner's model.pt (actor.py:50-72); retried while the file is being replaced."""
        path = self.model_path + 'model.pt'
        if not os.path.isfile(path):
            return
        for _ in range(20):
            try:
                model_dict = torch.load(path, map_location="cpu")
                weights = {name: model_dict[name] for name in ("actor", "target_actor", "critic", "target_critic")}
                break
            except Exception:
                sleep(np.random.rand() * 2 + 0.5)
        else:
            return
        self.weights = weights
        self.engine.load(weights)

    def _finish(self, done, seqs, states):
        """Pad, n-step rewards and priorities of the episodes of envs `done` (one batched call), memory.add, save."""
        from r2d2_b200 import actor_priority
        keep = [k for k in done if len(seqs[k]) >= self.sequence_length]
        if keep:
            for k in keep:                                                    # actor.py:173
                seqs[k].extend([(np.zeros(self.obs_size, np.float32), np.zeros(self.action_size, np.float32), [0.0], [1.0])
                                for _ in range(self.n_step)])
            episodes = [(np.stack([r[0] for r in seqs[k]]), np.stack([r[1] for r in seqs[k]]),
                         np.asarray([r[2][0] for r in seqs[k]], np.float32),
                         np.asarray([r[3][0] for r in seqs[k]], np.float32)) for k in keep]
            prios, rews = actor_priority.episode_priorities(
                self.weights["critic"], self.weights["target_actor"], self.weights["target_critic"], episodes,
                hidden=self.hidden, burn_in=self.burn_in_length, learning=self.learning_length, n_step=self.n_step,
                gamma=self.gamma, rewards_are_raw=True, device=self.device)
            for k, pr, rw in zip(keep, prios, rews):
                for i, row in enumerate(seqs[k]):
                    row[2][0] = float(rw[i])
                self.memory.add(seqs[k], states[k], [float(p) for p in pr])
        if len(self.memory.memory) > self.memory_save_interval:
            self.memory.save(self.actor_id)

    def run(self, max_episodes=None):
        """Step until `max_episodes` episodes (over all envs) have finished; forever for None."""
        n, A = self.n_envs, self.action_size
        obs = np.stack([get_obs(env.reset().observation)[0] for env in self.envs]).astype(np.float32)
        self.engine.reset()
        seqs, states = [[] for _ in range(n)], [[] for _ in range(n)]
        reward_sum = np.zeros(n)
        episode = step = 0
        while max_episodes is None or episode < max_episodes:
            mu, pre = self.engine.step(obs)                                   # pre-step states [4,2,n,H]
            action = np.clip(mu + np.random.normal(0, 0.3, (n, A)), -1, 1)
            nxt = obs.copy()
            done = []
            for k, env in enumerate(self.envs):
                reward = 0.0
                for _ in range(4):                                            # action repeat, actor.py:152-157
                    time_step = env.step(action[k])
                    reward += time_step.reward or 0.0
                    if time_step.last():
                        break
                nxt[k] = get_obs(time_step.observation)[0]
                last = time_step.last()
                reward_sum[k] += reward
                seqs[k].append((obs[k].copy(), action[k].astype(np.float32), [reward], [1.0 if last else 0.0]))
                st = pre[:, :, k].copy()
                states[k].append([[st[i, 0], st[i, 1]] for i in range(4)])
                if last:
                    done.append(k)
            step += 1
            if step % self.actor_parameter_update_interval == 0:
                self.load_model()
            if done:
                episode += len(done)
                if self.actor_id == 0:
                    print('episodes:', episode, 'step:', step, 'reward:', float(np.mean(reward_sum[done])))
                self._finish(done, seqs, states)
                mask = np.zeros(n, bool)
                for k in done:
                    nxt[k] = get_obs(self.envs[k].reset().observation)[0]
                    seqs[k], states[k] = [], []
                    reward_sum[k] = 0.0
                    mask[k] = True
                self.engine.reset(mask)
            obs = nxt
