"""Oracle harness: run the UNMODIFIED reference learner loop on CPU (this container only).

TEST INFRASTRUCTURE - never imported by the product path.  Only `oracle/make_golden.py`
(fixture generation) runs it, on a machine that has the reference sources (R2D2_REFERENCE_DIR).
Importing it needs no reference; the tests, smoke() and bench.py never call into it.

What it does (SURVEY.md section 8c / Appendix A):
  * puts stub modules for `dm_control`, `dm_control.suite`, `gym`, `PIL` in sys.modules
    (the reference imports them at learner.py:5-9 but uses only suite.load for sizes,
    learner.py:24-26);
  * makes `.cuda()` the identity on CPU (replay_memory.py:123-133, learner.py:39-41,100-101,119,
    models.py:35-36,78-79);
  * forces torch.load(weights_only=False) (memory{i}.pt is a pickle of deques/ndarrays,
    replay_memory.py:55-59);
  * writes a synthetic memory_data/memory0.pt in the actor file format (actor.py:163-176);
  * bounds the infinite `while True` (learner.py:78) by replacing `learner.time` (called once
    per iteration at learner.py:81) with a hook that records the previous iteration's locals
    and raises after N iterations; `learner.sleep` becomes a no-op;
  * optionally substitutes `models` by a hidden-size-parameterised restatement
    (oracle/ref_port.py nets) so cfg-2/cfg-3 (H != 128) can be driven by the real learner.py.
"""
from __future__ import annotations

import collections
import os
import sys
import types
from collections import OrderedDict

import numpy as np
import torch

from oracle import ref_port

REFERENCE_DIR = os.environ.get("R2D2_REFERENCE_DIR", "/root/reference")


class _StopLoop(Exception):
    pass


def reference_available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_DIR, "learner.py"))


def _install_stubs(obs_size: int, n_actions: int):
    class _Spec:
        shape = (n_actions,)

    class _TimeStep:
        observation = OrderedDict(o=np.zeros(obs_size, dtype=np.float32))

    class _Env:
        def action_spec(self):
            return _Spec()

        def reset(self):
            return _TimeStep()

    suite = types.ModuleType("dm_control.suite")
    suite.load = lambda domain_name=None, task_name=None: _Env()
    dmc = types.ModuleType("dm_control")
    dmc.suite = suite
    sys.modules["dm_control"] = dmc
    sys.modules["dm_control.suite"] = suite
    sys.modules.setdefault("gym", types.ModuleType("gym"))
    if "PIL" not in sys.modules:
        try:
            import PIL  # noqa: F401
            from PIL import Image  # noqa: F401
        except Exception:
            pil = types.ModuleType("PIL")
            pil.Image = types.ModuleType("PIL.Image")
            sys.modules["PIL"] = pil
            sys.modules["PIL.Image"] = pil.Image


def make_actor_file(path, **kw):
    """Synthetic memory{i}.pt in the actor format (oracle/ref_port.py synthetic_actor_file)."""
    torch.save(ref_port.synthetic_actor_file(**kw), path)


def run_reference_learner(*, obs_size, n_actions, hidden=128, batch_size=32, burn_in=20,
                          learning=40, n_step=5, n_iters=3, seed=1, data_seed=0,
                          n_episodes=None, episode_len=250, scratch=None, n_threads=None,
                          capture=True, models_module=None):
    """Run `n_iters` iterations of the real reference `Learner.run()`; return a list of
    per-iteration dicts of numpy arrays (batch, q, target, losses, grads, params, priorities)
    and the per-iteration wall times."""
    import tempfile
    import time as _time

    assert reference_available(), "reference not mounted; goldens can only be made in the build container"
    if n_threads:
        torch.set_num_threads(n_threads)
    seq_len = burn_in + learning
    if n_episodes is None:
        per_ep = episode_len + n_step - (seq_len + n_step - 1)
        n_episodes = (100 * batch_size + per_ep - 1) // per_ep + 1

    _install_stubs(obs_size, n_actions)
    ident = lambda self, *a, **k: self  # noqa: E731
    torch.Tensor.cuda = ident
    torch.nn.Module.cuda = ident
    if not getattr(torch.load, "_r2d2_patched", False):
        _orig_load = torch.load

        def _load(*a, **k):
            k.setdefault("weights_only", False)
            return _orig_load(*a, **k)

        _load._r2d2_patched = True
        torch.load = _load

    for m in ("learner", "actor", "replay_memory", "models", "utils"):
        sys.modules.pop(m, None)
    if models_module is not None:
        sys.modules["models"] = models_module
    if REFERENCE_DIR not in sys.path:
        sys.path.insert(0, REFERENCE_DIR)

    scratch = scratch or tempfile.mkdtemp(prefix="r2d2_ref_")
    os.makedirs(os.path.join(scratch, "model_data"), exist_ok=True)
    os.makedirs(os.path.join(scratch, "memory_data"), exist_ok=True)
    make_actor_file(os.path.join(scratch, "memory_data", "memory0.pt"), obs_size=obs_size,
                    n_actions=n_actions, hidden=hidden, n_episodes=n_episodes,
                    episode_len=episode_len, seed=data_seed, burn_in=burn_in, learning=learning,
                    n_step=n_step)
    cwd = os.getcwd()
    os.chdir(scratch)
    try:
        import learner as ref_learner  # the real /root/reference/learner.py

        torch.manual_seed(seed)
        lr = ref_learner.Learner(1)
        lr.batch_size = lr.memory.batch_size = batch_size
        lr.burn_in_length = lr.memory.burn_in_length = burn_in
        lr.learning_length = lr.memory.learning_length = learning
        lr.sequence_length = lr.memory.sequence_length = seq_len
        lr.n_step = lr.memory.n_step = n_step
        lr.model_save_interval = 10 ** 9
        lr.memory_update_interval = 10 ** 9

        records, stamps = [], []
        cur = {}

        def snap_params(net):
            return {k: v.detach().clone().numpy() for k, v in net.state_dict().items()}

        def snap_grads(net):
            return {k: p.grad.detach().clone().numpy() for k, p in net.named_parameters()}

        if capture:
            cur["actor_init"] = snap_params(lr.actor)
            cur["critic_init"] = snap_params(lr.critic)
            cur["target_actor_init"] = snap_params(lr.target_actor)
            cur["target_critic_init"] = snap_params(lr.target_critic)
            orig_sample = lr.memory.sample

            def sample_hook():
                out = orig_sample()
                cur["episode_index"] = np.asarray(out[0], dtype=np.int64)
                cur["sequence_index"] = np.asarray(out[1], dtype=np.int64)
                for name, t in zip(("obs", "act", "rew", "term", "a_state", "ta_state", "c_state", "tc_state"),
                                   out[2:]):
                    cur[name] = t.detach().clone().numpy()
                return out

            lr.memory.sample = sample_hook

            c_step, a_step = lr.critic_optimizer.step, lr.actor_optimizer.step

            def critic_step_hook(*a, **k):
                cur["critic_grad"] = snap_grads(lr.critic)
                r = c_step(*a, **k)
                cur["critic_after"] = snap_params(lr.critic)
                return r

            def actor_step_hook(*a, **k):
                cur["actor_grad"] = snap_grads(lr.actor)
                r = a_step(*a, **k)
                cur["actor_after"] = snap_params(lr.actor)
                return r

            lr.critic_optimizer.step = critic_step_hook
            lr.actor_optimizer.step = actor_step_hook

        def time_hook():
            stamps.append(_time.perf_counter())
            if capture and len(stamps) > 1:
                loc = sys._getframe(1).f_locals  # locals of Learner.run: previous iteration's values
                cur["q_value"] = loc["q_value"].detach().clone().numpy()
                cur["target_q_value"] = loc["target_q_value"].detach().clone().numpy()
                cur["critic_loss"] = np.float64(loc["critic_loss"].item())
                cur["actor_loss"] = np.float64(loc["actor_loss"].item())
                cur["average_td_loss"] = np.asarray(loc["average_td_loss"]).copy()
                ep, sq = cur["episode_index"], cur["sequence_index"]
                cur["priority_written"] = np.asarray(
                    [lr.memory.priority[int(e)][int(s)] for e, s in zip(ep, sq)], dtype=np.float64)
                cur["total_priority_written"] = np.asarray(
                    [lr.memory.total_priority[int(e)] for e in ep], dtype=np.float64)
                cur["target_actor_after"] = snap_params(lr.target_actor)
                cur["target_critic_after"] = snap_params(lr.target_critic)
                records.append(dict(cur))
                cur.clear()
            if len(stamps) > n_iters:
                raise _StopLoop()
            return stamps[-1]

        ref_learner.time = time_hook
        ref_learner.sleep = lambda *_a, **_k: None
        try:
            lr.run()
        except _StopLoop:
            pass
        times = np.diff(np.asarray(stamps))
        return records, times, lr
    finally:
        os.chdir(cwd)
        for m in ("learner", "actor", "replay_memory", "models", "utils"):
            sys.modules.pop(m, None)
        try:
            sys.path.remove(REFERENCE_DIR)
        except ValueError:
            pass


if __name__ == "__main__":
    recs, times, _ = run_reference_learner(obs_size=24, n_actions=6, n_iters=4)
    print("iter times (s):", np.round(times, 4))
    r = recs[0]
    print("keys:", sorted(r.keys()))
    print("q", r["q_value"].shape, "critic_loss", r["critic_loss"], "actor_loss", r["actor_loss"])
    print("prio", r["priority_written"][:4])
