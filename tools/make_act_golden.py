"""Generate tests/golden/ref_act_rollout.npz by executing the UNMODIFIED reference's acting loop on CPU.

Run where the reference sources are (R2D2_REFERENCE_DIR, as for oracle/make_golden.py):
    python tools/make_act_golden.py

  ref_act_rollout.npz   the real Actor.run() loop (actor.py:109-176) for one 64-step episode of a seeded synthetic env:
                        per step obs, the actor's un-noised output, the noisy action and the four recurrent states
                        recorded before the step; weight digests of the four nets (rebuilt by the tests from the torch
                        seed with the oracle/ref_port.py nets and checked bit for bit)

It uses the same harness pieces as oracle/make_golden.py's gen_actor_priorities: the stub modules of
oracle/ref_harness.py, `.cuda()` as the identity, no model.pt (load_model() is a no-op), the targets given their
own weights so that the fixture distinguishes the four roles.
"""
from __future__ import annotations

import collections
import os
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import ref_harness  # noqa: E402
from oracle.make_golden import OUT, array_digest  # noqa: E402


class _ActEnv:
    """Seeded synthetic environment with the dm_control TimeStep surface the reference's Actor.run() reads
    (reset / step / last / observation / reward); the episode ends after 4 * steps environment steps."""

    class _TS:
        def __init__(self, obs, reward, last):
            self.observation, self.reward, self._last = collections.OrderedDict(o=obs), reward, last

        def last(self):
            return self._last

    def __init__(self, obs_size, n_actions, steps, seed):
        self.rng = np.random.default_rng(seed)
        self.obs_size, self.n_actions, self.steps = obs_size, n_actions, steps
        self.A = (self.rng.standard_normal((obs_size, obs_size)) * 0.3).astype(np.float32)
        self.Bm = (self.rng.standard_normal((n_actions, obs_size)) * 0.8).astype(np.float32)

    def action_spec(self):
        return type("Spec", (), {"shape": (self.n_actions,)})()

    def reset(self):
        self.t = 0
        self.x = self.rng.standard_normal(self.obs_size).astype(np.float32)
        return self._TS(self.x, 0.0, False)

    def step(self, action):
        self.t += 1
        self.x = np.tanh(self.x @ self.A + np.asarray(action, np.float32) @ self.Bm).astype(np.float32)
        return self._TS(self.x, float(-np.square(self.x).mean()), self.t >= 4 * self.steps)


class _StopActor(Exception):
    pass


def gen_act_rollout(O=17, A=6, steps=64, seed=300, env_seed=301, noise_seed=302):
    """The real Actor.run() loop (actor.py:109-176) for one episode of `steps` steps: per step the observation, the
    actor's un-noised output mu, the noisy clipped action and the four recurrent states recorded BEFORE the step
    (actor.py:136-139,166-167).  Pins the net order, the critics' input (mu, not the noisy action) and the zero state
    at episode start for the batched acting kernels (r2d2_act_*)."""
    assert ref_harness.reference_available(), "reference not mounted; the fixture can only be made where it is"
    ref_harness._install_stubs(O, A)
    ident = lambda self, *a, **k: self  # noqa: E731
    torch.Tensor.cuda = ident
    torch.nn.Module.cuda = ident
    for m in ("actor", "replay_memory", "models", "utils", "learner"):
        sys.modules.pop(m, None)
    if ref_harness.REFERENCE_DIR not in sys.path:
        sys.path.insert(0, ref_harness.REFERENCE_DIR)
    cwd = os.getcwd()
    os.chdir(tempfile.mkdtemp(prefix="r2d2_act_"))          # no model_data/model.pt: load_model() is a no-op
    try:
        import actor as ref_actor
        import models as ref_models
        ref_actor.sleep = lambda *_a, **_k: None
        torch.manual_seed(seed)
        a = ref_actor.Actor(0)
        a.target_actor = ref_models.ActorNet(O, A, 0).eval()     # own weights for the targets
        a.target_critic = ref_models.CriticNet(O, A, 0).eval()
        a.env = _ActEnv(O, A, steps, env_seed)
        mus = []
        net = a.actor

        class _Recorded:                                       # the actor's own call, its output recorded
            def __call__(self, x):
                y = net(x)
                mus.append(y.detach().numpy()[0].copy())
                return y

            def __getattr__(self, name):
                return getattr(net, name)

        a.actor = _Recorded()
        a.memory.add = lambda *_a, **_k: (_ for _ in ()).throw(_StopActor())   # stop after the first episode
        np.random.seed(noise_seed)
        try:
            with torch.no_grad():
                a.run()
        except _StopActor:
            pass
        n_real = len(a.recurrent_state)
        assert n_real == steps, n_real
        d = {"torch_version": np.array(torch.__version__), "seed": np.int64(seed), "env_seed": np.int64(env_seed),
             "noise_seed": np.int64(noise_seed), "cfg": np.int64([O, A, 128, steps])}
        for name in ("actor", "target_actor", "critic", "target_critic"):
            m = net if name == "actor" else getattr(a, name)
            for k, v in m.state_dict().items():
                d[f"{name}/{k}"] = np.array(array_digest(v.detach().numpy()))
        d["obs"] = np.stack([r[0] for r in a.sequence[:n_real]]).astype(np.float32)
        d["action"] = np.stack([r[1] for r in a.sequence[:n_real]]).astype(np.float64)
        d["mu"] = np.stack(mus).astype(np.float32)
        d["states"] = np.asarray(a.recurrent_state, np.float32)         # [steps, 4, 2, H]
        d["reward"] = np.asarray([r[2][0] for r in a.sequence[:n_real]], np.float64)
    finally:
        os.chdir(cwd)
        for m in ("actor", "replay_memory", "models", "utils"):
            sys.modules.pop(m, None)
    path = os.path.join(OUT, "ref_act_rollout.npz")
    np.savez_compressed(path, **d)
    print("ref_act_rollout.npz ok", os.path.getsize(path))


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(8)
    gen_act_rollout()
