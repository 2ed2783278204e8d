"""Batched GPU acting (r2d2_act_*, r2d2_b200.acting.ActEngine, actor.VecActor) against the reference's acting loop
(/root/reference/actor.py:136-148): one step of actor, target actor, critic(x, mu), target critic(x, mu_t) with the
four (h, c) states recorded before the step.

 * CPU: the float64 restatement (oracle/learner_oracle.net_forward, one step at a time, the reference's call order)
   reproduces tests/golden/ref_act_rollout.npz (the unmodified Actor.run() loop, tools/make_act_golden.py);
   r2d2_act_create validates its arguments before any CUDA call.
 * GPU: ActEngine against that fixture and against the float64 oracle free-running at every batch-tile edge with
   four different weight sets, staggered resets and a mid-rollout reload; saturated gates; VecActor against the
   drop-in CPU Actor and per env against the oracle; the saved actor file through LearnerReplayMemory.load.
"""
import os
import sys

import numpy as np
import pytest

from conftest import checked_state, load_golden, rel_l2

NETS = ("actor", "target_actor", "critic", "target_critic")
SHAPES = ((3, 1), (17, 6), (376, 17))        # BASELINE.json (obs, act) shapes
BATCHES = (1, 2, 15, 16, 17, 63, 64, 65, 255, 256, 257, 1000)


# ---------------------------------------------------------------------------------------------- float64 oracle
def oracle_step(P, x, st):
    """One acting step in float64 with oracle/learner_oracle.net_forward: P {net: state_dict of arrays}, x [B,O],
    st [4,2,B,H] -> (mu [B,A], new state [4,2,B,H]); the critics get the un-noised mu and mu_t."""
    from oracle import learner_oracle as lo
    x = np.asarray(x, np.float64)
    new = np.empty(st.shape, np.float64)

    def cell(i, inp, critic):
        sv = lo.net_forward(P[NETS[i]], inp[None], st[i, 0], st[i, 1], critic=critic)
        new[i, 0], new[i, 1] = sv["hs"][1], sv["cs"][1]
        return sv["out"][0]

    mu = cell(0, x, False)                                   # actor(x)             actor.py:141
    mu_t = cell(1, x, False)                                 # target_actor(x)      actor.py:142
    cell(2, np.concatenate([x, mu], 1), True)                # critic(x, mu)        actor.py:143
    cell(3, np.concatenate([x, mu_t], 1), True)              # target_critic(x, mu_t) actor.py:144
    return mu, new


def f64(sd):
    return {k: np.asarray(v.detach().numpy() if hasattr(v, "detach") else v, np.float64) for k, v in sd.items()}


def fixture_nets(g):
    """The reference's four nets: under its torch seed Actor() builds actor, critic; then the fixture's own target
    actor, target critic.  The port's nets draw the same weights (digests checked)."""
    import torch
    from oracle import ref_port
    O, A, H, _ = (int(v) for v in g["cfg"])
    torch.manual_seed(int(g["seed"]))
    made = {"actor": ref_port.PortActorNet(O, A, 0, H), "critic": ref_port.PortCriticNet(O, A, 0, H),
            "target_actor": ref_port.PortActorNet(O, A, 0, H), "target_critic": ref_port.PortCriticNet(O, A, 0, H)}
    return {n: checked_state(g, n, made[n]) for n in NETS}


def random_nets(O, A, H, seed, scale=1.0):
    """Four different weight sets.  The head is far larger than the reference's +-3e-3 init so that mu matters to
    the critics: feeding them the wrong action, or swapping roles, changes their states."""
    rng = np.random.default_rng(seed)
    out = {}
    for i, n in enumerate(NETS):
        I = O + (A if i >= 2 else 0)
        u = lambda shape, b: rng.uniform(-b, b, shape).astype(np.float32)  # noqa: E731
        out[n] = {"l1.weight": u((H, I), 1.5 / np.sqrt(I)), "l1.bias": u((H,), 0.1),
                  "l2.weight_ih": u((4 * H, H), scale * 1.5 / np.sqrt(H)),
                  "l2.weight_hh": u((4 * H, H), scale * 1.5 / np.sqrt(H)),
                  "l2.bias_ih": u((4 * H,), 0.1), "l2.bias_hh": u((4 * H,), 0.1),
                  "l3.weight": u((A, H), 2.0 / np.sqrt(H)), "l3.bias": u((A,), 0.1)}
    return out


# ---------------------------------------------------------------------------------------------- CPU
def test_oracle_reproduces_reference_act_rollout():
    g = load_golden("ref_act_rollout.npz")
    P = {n: f64(sd) for n, sd in fixture_nets(g).items()}
    O, A, H, steps = (int(v) for v in g["cfg"])
    assert g["obs"].shape == (steps, O) and g["states"].shape == (steps, 4, 2, H)
    assert not g["states"][0].any()                          # zero state at episode start (models.py:34-36)
    st = np.zeros((4, 2, 1, H))
    for t in range(steps):
        rec = g["states"][t].astype(np.float64)
        assert rel_l2(st[:, :, 0], rec) < 2e-5, (t, rel_l2(st[:, :, 0], rec))    # states recorded BEFORE step t
        mu, st = oracle_step(P, g["obs"][t][None], st)
        assert rel_l2(mu[0], g["mu"][t]) < 2e-5, (t, rel_l2(mu[0], g["mu"][t]))
    # the noisy action is mu + N(0, 0.3) clipped (actor.py:146-148), under the fixture's numpy seed
    rs = np.random.RandomState(int(g["noise_seed"]))
    for t in range(steps):
        a = np.clip(g["mu"][t].astype(np.float64) + rs.normal(0, 0.3, A), -1, 1)
        assert np.allclose(a, g["action"][t], atol=1e-6)


def test_oracle_critics_see_mu_not_the_noisy_action():
    """The fixture distinguishes feeding the critic mu from feeding it the noisy action it stores."""
    from oracle import learner_oracle as lo
    g = load_golden("ref_act_rollout.npz")
    P = {n: f64(sd) for n, sd in fixture_nets(g).items()}
    H = int(g["cfg"][2])
    h, c = np.zeros((1, H)), np.zeros((1, H))
    x = np.concatenate([g["obs"][0], g["action"][0]])[None].astype(np.float64)
    sv = lo.net_forward(P["critic"], x[None], h, c, critic=True)
    assert rel_l2(sv["hs"][1], g["states"][1, 2, 0]) > 1e-3


def test_act_create_rejects_unsupported_shapes():
    from ctypes import c_void_p

    from r2d2_b200 import native as nv
    lib = nv.lib()
    h = c_void_p()
    for (O, A, H, B), rc in (((17, 6, 48, 4), -3), ((17, 6, 16, 4), -3), ((17, 6, 544, 4), -3), ((17, 6, 0, 4), -3),
                             ((17, 0, 128, 4), -3), ((17, 33, 128, 4), -3), ((0, 6, 128, 4), -2),
                             ((17, 6, 128, 0), -2), ((17, 6, 128, -5), -2)):
        got = lib.r2d2_act_create(nv.byref(h), nv.byref(nv.NetShape(O, A, H, 0)), B)
        assert got == rc, ((O, A, H, B), got, lib.r2d2_last_error())
        assert lib.r2d2_last_error(), (O, A, H, B)
        assert not h.value
    assert lib.r2d2_act_create(None, nv.byref(nv.NetShape(17, 6, 128, 0)), 4) == -2
    assert lib.r2d2_act_create(nv.byref(h), None, 4) == -2


# ---------------------------------------------------------------------------------------------- GPU helpers
def row_compare(name, x, ref, tol_g=1e-3, tol_r=5e-3):
    """Global relative L2 and the worst batch row against the RMS row norm (batch axis = last but one)."""
    x, ref = np.asarray(x, np.float64), np.asarray(ref, np.float64)
    B = ref.shape[-2]
    dx = np.moveaxis(x - ref, -2, 0).reshape(B, -1)
    nref = max(float(np.linalg.norm(ref)), 1e-30)
    rows = np.linalg.norm(dx, axis=1) / (nref / np.sqrt(B))
    b = int(np.nanargmax(rows)) if np.isfinite(rows).all() else int(np.argmax(~np.isfinite(rows)))
    g = float(np.linalg.norm(dx) / nref)
    ok = g <= tol_g and rows[b] <= tol_r
    return ok, f"{name}: global {g:.2e} (tol {tol_g}), worst row b={b} {rows[b]:.2e} (tol {tol_r})"


class _Acc:
    """Per-row squared error and reference norm summed over steps, per tensor."""

    def __init__(self):
        self.d = {}

    def add(self, name, x, ref):
        x, ref = np.asarray(x, np.float64), np.asarray(ref, np.float64)
        B = ref.shape[-2]
        e = np.square(np.moveaxis(x - ref, -2, 0).reshape(B, -1)).sum(1)
        r = float(np.square(ref).sum())
        if name in self.d:
            self.d[name][0] += e
            self.d[name][1] += r
        else:
            self.d[name] = [e, r]

    def failures(self, tol_g=1e-3, tol_r=5e-3):
        bad, worst = [], 0.0
        for name, (e, r) in self.d.items():
            B = e.size
            nref = max(np.sqrt(r), 1e-30)
            rows = np.sqrt(e) / (nref / np.sqrt(B))
            g = float(np.sqrt(e.sum()) / nref)
            b = int(np.nanargmax(rows)) if np.isfinite(rows).all() else int(np.argmax(~np.isfinite(rows)))
            worst = max(worst, g)
            if not (g <= tol_g and rows[b] <= tol_r):
                bad.append(f"{name}: global {g:.2e}, worst row b={b} {rows[b]:.2e}")
        return bad, worst


def _engine(O, A, H, B):
    from r2d2_b200.acting import ActEngine
    return ActEngine(O, A, H, B, device="cuda:0")


# ---------------------------------------------------------------------------------------------- GPU: ActEngine
@pytest.mark.gpu
def test_gpu_engine_reproduces_reference_act_rollout():
    g = load_golden("ref_act_rollout.npz")
    nets = fixture_nets(g)
    O, A, H, steps = (int(v) for v in g["cfg"])
    eng = _engine(O, A, H, 1)
    eng.load(nets)
    eng.reset()
    mus, states = [], []
    for t in range(steps):
        mu, st = eng.step(g["obs"][t][None])
        mus.append(mu[0])
        states.append(st[:, :, 0])
    assert not np.asarray(states[0]).any()
    assert rel_l2(np.asarray(mus), g["mu"]) < 1e-3, rel_l2(np.asarray(mus), g["mu"])
    states = np.asarray(states)
    for i, n in enumerate(NETS):
        for j, hc in enumerate("hc"):
            e = rel_l2(states[1:, i, j], g["states"][1:, i, j])
            assert e < 1e-3, (n, hc, e)
    assert eng.status() == 0
    eng.close()


def _free_running(H, B, O, A, steps=100, seed=0):
    """ActEngine against the float64 oracle for `steps` steps with staggered per-env resets and a reload of new
    weights half way; every step checks mu and the four (h, c) of every env."""
    rng = np.random.default_rng(seed)
    nets = random_nets(O, A, H, seed)
    nets2 = random_nets(O, A, H, seed + 1)
    P, P2 = ({n: f64(sd) for n, sd in w.items()} for w in (nets, nets2))
    eng = _engine(O, A, H, max(B, 3))
    eng.load(nets)
    eng.reset()
    st = np.zeros((4, 2, B, H))
    acc = _Acc()
    period = 23 + (seed % 7)
    for t in range(steps):
        if t == steps // 2:
            eng.load(nets2)
            P = P2
        if t > 0:
            mask = ((np.arange(B) * 7 + t) % period) == 0            # staggered episode starts
            if mask.any():
                eng.reset(mask)
                st[:, :, mask] = 0.0
        x = rng.standard_normal((B, O)).astype(np.float32)
        mu, pre = eng.step(x)
        if t < 3 or t == steps // 2:
            ok, msg = row_compare(f"recorded state t={t}", pre, st)
            assert ok, msg
        mu_ref, st = oracle_step(P, x, st)
        acc.add("mu", mu, mu_ref)
        post = eng.state()
        for i, n in enumerate(NETS):
            acc.add(f"{n}.h", post[i, 0], st[i, 0])
            acc.add(f"{n}.c", post[i, 1], st[i, 1])
        st = st.astype(np.float64)
    bad, worst = acc.failures()
    status = eng.status()
    eng.close()
    return bad, worst, status


@pytest.mark.gpu
@pytest.mark.parametrize("H", (32, 64, 128, 256, 512))
def test_gpu_engine_free_running_vs_oracle(H):
    bad_all = []
    for i, B in enumerate(BATCHES):
        O, A = SHAPES[(i + H // 32) % len(SHAPES)]
        steps = 100 if H * B <= 256 * 257 else 40
        bad, worst, status = _free_running(H, B, O, A, steps=steps, seed=H + B)
        assert status == 0, (H, B, "bounded mbarrier wait expired")
        bad_all += [f"H={H} B={B} O={O} A={A}: {m}" for m in bad]
    assert not bad_all, "\n".join(bad_all)


@pytest.mark.gpu
@pytest.mark.parametrize("H,B", ((128, 17), (512, 65)))
def test_gpu_engine_saturated_gates(H, B):
    O, A = 17, 6
    nets = random_nets(O, A, H, 99, scale=80.0)
    P = {n: f64(sd) for n, sd in nets.items()}
    eng = _engine(O, A, H, B)
    eng.load(nets)
    eng.reset()
    rng = np.random.default_rng(5)
    st = np.zeros((4, 2, B, H))
    peak = 0.0
    for t in range(20):
        x = (rng.standard_normal((B, O)) * 100).astype(np.float32)
        mu, _ = eng.step(x)
        # pre-activations of the gates (what the kernel sees) reach +-60 and beyond
        z = np.tanh(x.astype(np.float64) @ P["actor"]["l1.weight"].T + P["actor"]["l1.bias"])
        peak = max(peak, float(np.abs(z @ P["actor"]["l2.weight_ih"].T).max()))
        mu_ref, st = oracle_step(P, x, st)
        post = eng.state()
        assert np.isfinite(mu).all() and np.isfinite(post).all(), t
        assert np.abs(mu - mu_ref).max() < 1e-2, (t, np.abs(mu - mu_ref).max())
        cmax = max(1.0, float(np.abs(st[:, 1]).max()))
        assert np.abs(post[:, 0] - st[:, 0]).max() < 2e-2, (t, np.abs(post[:, 0] - st[:, 0]).max())
        assert np.abs(post[:, 1] - st[:, 1]).max() < 2e-2 * cmax, (t, np.abs(post[:, 1] - st[:, 1]).max(), cmax)
        st = post.astype(np.float64)          # follow the kernel: bound the error of one step, not of a chaotic chain
    assert peak >= 60.0, peak
    assert eng.status() == 0
    eng.close()


@pytest.mark.gpu
def test_gpu_engine_rejects_bad_steps():
    from r2d2_b200 import native as nv
    eng = _engine(17, 6, 64, 8)
    with pytest.raises(nv.NativeError):
        eng.step(np.zeros((2, 17), np.float32))             # no weights loaded
    eng.load(random_nets(17, 6, 64, 1))
    with pytest.raises(nv.NativeError):
        eng.step(np.zeros((9, 17), np.float32))             # more envs than max_batch
    with pytest.raises(nv.NativeError):
        eng.step(np.zeros((2, 16), np.float32))
    assert eng.status() == 0
    eng.close()


# ---------------------------------------------------------------------------------------------- GPU: VecActor
def _dropin(monkeypatch, O, A, H):
    monkeypatch.setenv("R2D2_OBS_SIZE", str(O))
    monkeypatch.setenv("R2D2_N_ACTIONS", str(A))
    monkeypatch.setenv("R2D2_HIDDEN", str(H))
    monkeypatch.delenv("R2D2_ACTOR_DEVICE", raising=False)
    for m in ("actor", "learner", "replay_memory", "models", "utils"):
        sys.modules.pop(m, None)
    import actor as dropin_actor
    return dropin_actor


def _write_model(path, nets):
    import torch
    torch.save({n: {k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in sd.items()} for n, sd in nets.items()}, path)


def _recording(mem):
    """Record every episode handed to memory.add and the episode lengths of every save."""
    added, saved = [], []
    add, save = mem.add, mem.save

    def rec_add(seq, states, prio):
        added.append((seq, states, list(prio)))
        add(seq, states, prio)

    def rec_save(aid):
        saved.append([len(e) for e in mem.memory])
        save(aid)
    mem.add, mem.save = rec_add, rec_save
    return added, saved


@pytest.mark.gpu
def test_gpu_vec_actor_one_env_matches_cpu_actor(monkeypatch, tmp_path):
    import torch
    O, A, H = 17, 6, 128
    dropin = _dropin(monkeypatch, O, A, H)
    monkeypatch.chdir(tmp_path)
    os.makedirs("model_data")
    os.makedirs("memory_data")
    nets = random_nets(O, A, H, 7)
    _write_model("model_data/model.pt", nets)
    runs = {}
    for kind in ("cpu", "vec"):
        torch.manual_seed(0)
        a = dropin.Actor(3) if kind == "cpu" else dropin.VecActor(3, 1)
        for env in ([a.env] if kind == "cpu" else a.envs):
            env.episode_len = 70
        added, _ = _recording(a.memory)
        np.random.seed(11)
        a.run(max_episodes=1)
        assert len(added) == 1
        runs[kind] = added[0]
        if kind == "vec":
            assert a.engine.status() == 0
    (s_c, st_c, p_c), (s_v, st_v, p_v) = runs["cpu"], runs["vec"]
    assert len(s_c) == len(s_v) == 70 + 5 and len(st_c) == len(st_v) == 70
    for i in range(4):                                   # obs, action, n-step reward, terminal
        a_c = np.asarray([np.asarray(r[i], np.float64).reshape(-1) for r in s_c])
        a_v = np.asarray([np.asarray(r[i], np.float64).reshape(-1) for r in s_v])
        assert np.abs(a_c - a_v).max() < (1e-4 if i < 2 else 1e-3 * max(1.0, np.abs(a_c).max())), (i, np.abs(a_c - a_v).max())
    sc, sv = np.asarray(st_c, np.float64), np.asarray(st_v, np.float64)     # [steps, 4, 2, H]
    assert not sv[0].any()
    for i, n in enumerate(NETS):
        for j, hc in enumerate("hc"):
            assert rel_l2(sv[:, i, j], sc[:, i, j]) < 1e-3, (n, hc, rel_l2(sv[:, i, j], sc[:, i, j]))
    assert len(p_c) == len(p_v) == 70 - 60
    assert rel_l2(p_v, p_c) < 1e-3, rel_l2(p_v, p_c)


@pytest.mark.gpu
def test_gpu_vec_actor_eight_envs_vs_oracle_and_learner_ingest(monkeypatch, tmp_path):
    O, A, H, n = 17, 6, 64, 8
    dropin = _dropin(monkeypatch, O, A, H)
    monkeypatch.chdir(tmp_path)
    os.makedirs("model_data")
    os.makedirs("memory_data")
    nets = random_nets(O, A, H, 21)
    _write_model("model_data/model.pt", nets)
    P = {k: f64(sd) for k, sd in nets.items()}
    va = dropin.VecActor(0, n)
    lens = [61 + 5 * k for k in range(n)]                 # every env ends its episode at a different step
    for env, L in zip(va.envs, lens):
        env.episode_len = L
    added, saved = _recording(va.memory)
    np.random.seed(3)
    va.run(max_episodes=n)
    assert va.engine.status() == 0
    assert sorted(len(st) for _, st, _ in added) == lens
    for seq, states, prio in added:
        E = len(states)
        assert len(seq) == E + 5 and len(prio) == E - 60
        obs = np.stack([r[0] for r in seq[:E]])
        rec = np.asarray(states, np.float64)              # [E, 4, 2, H]
        assert not rec[0].any()                           # zero state at episode start
        st = np.zeros((4, 2, 1, H))
        ref = []
        for t in range(E):
            ref.append(st[:, :, 0])
            _, st = oracle_step(P, obs[t][None], st)
        ref = np.asarray(ref)
        for i, net in enumerate(NETS):
            for j, hc in enumerate("hc"):
                assert rel_l2(rec[:, i, j], ref[:, i, j]) < 1e-3, (E, net, hc, rel_l2(rec[:, i, j], ref[:, i, j]))
    # the last actor file ingests through the drop-in learner memory with the reference's sequence count
    assert saved and os.path.isfile("memory_data/memory0.pt")
    sys.modules.pop("replay_memory", None)
    import replay_memory
    lm = replay_memory.LearnerReplayMemory(memory_sequence_size=10 ** 6, batch_size=4, hidden=H)
    lm.load(0)
    assert lm.sequence_counter == sum(L - (60 + 5 - 1) for L in saved[-1]), (lm.sequence_counter, saved[-1])
    assert len(lm.memory) == len(saved[-1])


def test_actor_process_without_envs_variable_is_the_cpu_actor(monkeypatch):
    """R2D2_ACTOR_ENVS unset: actor_process builds the drop-in CPU Actor, as before."""
    dropin = _dropin(monkeypatch, 5, 2, 32)
    monkeypatch.delenv("R2D2_ACTOR_ENVS", raising=False)
    made = []

    class _Stop(Exception):
        pass

    def fake_run(self, *a, **k):
        made.append(type(self).__name__)
        raise _Stop()
    monkeypatch.setattr(dropin.Actor, "run", fake_run)
    monkeypatch.setattr(dropin.VecActor, "run", fake_run)
    with pytest.raises(_Stop):
        dropin.actor_process(0)
    assert made == ["Actor"]
