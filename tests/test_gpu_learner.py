"""End-to-end parity of the native learner iteration (learner.py:84-139) on the GPU.

 * against fixtures produced by the UNMODIFIED reference (tests/golden/ref_*.npz, oracle/make_golden.py):
   same sampled batch, same initial weights -> q, target, losses, gradients, post-Adam weights and
   priorities within 1e-3 relative (north_star tolerance; relative L2 per tensor, see SURVEY section 7 on
   why element-wise relative error is ill-posed where |q| -> 0);
 * at BASELINE.json configs[1] size (obs=17 act=6 hidden=256 seq_len=80 burn_in=40 batch=256) against
   the CPU port of the reference (oracle/ref_port.py) on the same synthetic batch.
"""
import numpy as np
import pytest
import torch

from conftest import golden_batch, golden_init, golden_sample, load_golden, rel_l2
from oracle import ref_port

pytestmark = pytest.mark.gpu

TOL = 1e-3  # north_star: "within 1e-3 relative on the same sampled batch"


@pytest.fixture(scope="module")
def eng_mod():
    from r2d2_b200 import engine
    return engine


def _cfg(eng_mod, g):
    return eng_mod.PathConfig(obs=int(g["cfg/obs_size"]), act=int(g["cfg/n_actions"]), hidden=int(g["cfg/hidden"]),
                              batch=int(g["cfg/batch_size"]), burn_in=int(g["cfg/burn_in"]),
                              learning=int(g["cfg/learning"]), n_step=int(g["cfg/n_step"]))


def flat_sd(views):
    return {k: v.detach().cpu().numpy() for k, v in views.items()}


@pytest.mark.parametrize("name", ["ref_walker_h128.npz", "ref_pend_h128.npz", "ref_tiny_h32.npz"])
def test_against_reference_goldens(eng_mod, name):
    g = load_golden(name)
    cfg = _cfg(eng_mod, g)
    eng = eng_mod.LearnerEngine(cfg)
    eng.load_state_dicts(*golden_init(g))
    report = []
    for it in range(int(g["n_iters"])):
        eng.set_batch(golden_batch(g, it))
        # gradients are overwritten by the next phase only for the same net, so read them after the step
        eng.step()
        torch.cuda.synchronize()
        errs = {
            "q": rel_l2(eng.q_value.cpu().numpy(), g[f"it{it}/q_value"]),
            "target": rel_l2(eng.target_q_value.cpu().numpy(), g[f"it{it}/target_q_value"]),
            "td": rel_l2(eng.td_sq.cpu().numpy(), g[f"it{it}/average_td_loss"]),
            "prio": rel_l2(eng.priority.cpu().numpy(), g[f"it{it}/priority_written"]),
            "critic_loss": abs(eng.losses[0].item() - float(g[f"it{it}/critic_loss"])) / abs(float(g[f"it{it}/critic_loss"])),
            "actor_loss": abs(eng.losses[1].item() - float(g[f"it{it}/actor_loss"])) / max(abs(float(g[f"it{it}/actor_loss"])), 1e-12),
        }
        for net in ("actor", "critic"):
            gr, pa = flat_sd(eng.views(net, "grads")), flat_sd(eng.views(net))
            for k in eng_mod.PARAM_KEYS:
                gn = float(g[f"it{it}/{net}_grad_norm/{k}"])
                errs[f"{net}_gnorm/{k}"] = abs(np.linalg.norm(gr[k].astype(np.float64)) - gn) / max(gn, 1e-30)
                errs[f"{net}_after_sub/{k}"] = rel_l2(pa[k].reshape(-1)[::97], g[f"it{it}/{net}_after_sub/{k}"])
                if it == 0:
                    errs[f"{net}_grad/{k}"] = rel_l2(golden_sample(g, 0, net, k, gr[k]), g[f"it0/{net}_grad/{k}"])
                    errs[f"{net}_after/{k}"] = rel_l2(golden_sample(g, 0, net, k, pa[k]), g[f"it0/{net}_after/{k}"])
        report.append(errs)
        bad = {k: v for k, v in errs.items() if not v < TOL}
        assert not bad, f"{name} iteration {it}: {bad}"
    worst = max(max(e.values()) for e in report)
    print(f"{name}: worst relative error over {len(report)} iterations = {worst:.3e}")


def test_cfg2_full_size_against_port(eng_mod):
    """BASELINE.json configs[1]: obs=17 act=6 hidden=256 seq_len=80 burn_in=40 batch=256."""
    pc = ref_port.PathConfig(obs=17, act=6, hidden=256, batch=256, burn_in=40, learning=80, n_step=5)
    torch.set_num_threads(max(1, min(32, torch.get_num_threads())))
    port = ref_port.PortLearner(pc, seed=1)
    cfg = eng_mod.PathConfig(obs=17, act=6, hidden=256, batch=256, burn_in=40, learning=80, n_step=5)
    eng = eng_mod.LearnerEngine(cfg)
    sd = lambda m: {k: v.detach().numpy() for k, v in m.state_dict().items()}  # noqa: E731
    eng.load_state_dicts(sd(port.actor), sd(port.critic))
    for it in range(2):
        batch = ref_port.synthetic_batch(pc, seed=it)
        ref = port.iteration(batch)
        eng.set_batch(batch)
        eng.step()
        torch.cuda.synchronize()
        errs = {"q": rel_l2(eng.q_value.cpu().numpy(), ref["q_value"]),
                "target": rel_l2(eng.target_q_value.cpu().numpy(), ref["target_q_value"]),
                "prio": rel_l2(eng.priority.cpu().numpy(), ref["priority"]),
                "critic_loss": abs(eng.losses[0].item() - ref["critic_loss"]) / abs(ref["critic_loss"]),
                "actor_loss": abs(eng.losses[1].item() - ref["actor_loss"]) / abs(ref["actor_loss"])}
        for net in ("actor", "critic"):
            gr, pa = flat_sd(eng.views(net, "grads")), flat_sd(eng.views(net))
            for k in eng_mod.PARAM_KEYS:
                errs[f"{net}_grad/{k}"] = rel_l2(gr[k], ref[f"{net}_grad"][k])
                errs[f"{net}_after/{k}"] = rel_l2(pa[k], ref[f"{net}_after"][k])
        bad = {k: v for k, v in errs.items() if not v < TOL}
        assert not bad, f"iteration {it}: {bad}"
        print(f"cfg-2 iteration {it}: worst relative error {max(errs.values()):.3e}")


@pytest.mark.parametrize("batch", [24, 512])
def test_cfg3_hidden_512_against_port(eng_mod, batch):
    """BASELINE.json configs[2] (obs=376 act=17 hidden=512 seq_len=80 burn_in=40): the cluster-of-16 tcgen05 scan
    (W_hh hi plane in tensor memory, lo plane split between tensor and shared memory) at the full batch of 512 and at a
    batch that fills a single 16-row tile, against the CPU port of the reference on the same synthetic batch."""
    import ctypes
    from r2d2_b200 import native as nv
    pc = ref_port.PathConfig(obs=376, act=17, hidden=512, batch=batch, burn_in=40, learning=80, n_step=5)
    torch.set_num_threads(max(1, min(32, torch.get_num_threads())))
    port = ref_port.PortLearner(pc, seed=2)
    cfg = eng_mod.PathConfig(obs=376, act=17, hidden=512, batch=batch, burn_in=40, learning=80, n_step=5)
    eng = eng_mod.LearnerEngine(cfg)
    sd = lambda m: {k: v.detach().numpy() for k, v in m.state_dict().items()}  # noqa: E731
    eng.load_state_dicts(sd(port.actor), sd(port.critic))
    batch_np = ref_port.synthetic_batch(pc, seed=4)
    ref = port.iteration(batch_np)
    eng.set_batch(batch_np)
    eng.step()
    torch.cuda.synchronize()
    status = ctypes.c_int(0)
    nv.check(nv.lib().r2d2_scan_status(ctypes.byref(status), nv.current_stream()))
    assert status.value == 0, f"a bounded mbarrier wait timed out inside a scan kernel (code {status.value})"
    errs = {"q": rel_l2(eng.q_value.cpu().numpy(), ref["q_value"]),
            "target": rel_l2(eng.target_q_value.cpu().numpy(), ref["target_q_value"]),
            "prio": rel_l2(eng.priority.cpu().numpy(), ref["priority"]),
            "critic_loss": abs(eng.losses[0].item() - ref["critic_loss"]) / abs(ref["critic_loss"]),
            "actor_loss": abs(eng.losses[1].item() - ref["actor_loss"]) / abs(ref["actor_loss"])}
    for net in ("actor", "critic"):
        gr, pa = flat_sd(eng.views(net, "grads")), flat_sd(eng.views(net))
        for k in eng_mod.PARAM_KEYS:
            errs[f"{net}_grad/{k}"] = rel_l2(gr[k], ref[f"{net}_grad"][k])
            errs[f"{net}_after/{k}"] = rel_l2(pa[k], ref[f"{net}_after"][k])
    bad = {k: v for k, v in errs.items() if not v < TOL}
    assert not bad, bad
    print(f"cfg-3 batch {batch}: worst relative error {max(errs.values()):.3e}")


def test_hard_target_update(eng_mod):
    cfg = eng_mod.PathConfig(obs=5, act=2, hidden=32, batch=4, burn_in=3, learning=4, n_step=2, target_interval=2)
    pc = ref_port.PathConfig(obs=5, act=2, hidden=32, batch=4, burn_in=3, learning=4, n_step=2, target_interval=2)
    eng = eng_mod.LearnerEngine(cfg)
    before = eng.flat["target_critic"].clone()
    for it in range(2):
        eng.set_batch(ref_port.synthetic_batch(pc, seed=it))
        eng.step()
        torch.cuda.synchronize()
        if it == 0:
            assert torch.equal(eng.flat["target_critic"], before)       # step 1: no copy (learner.py:131)
    assert eng.step_count == 2
    assert torch.equal(eng.flat["target_critic"], eng.flat["critic"])   # step 2: hard copy (learner.py:63-65)
    assert torch.equal(eng.flat["target_actor"], eng.flat["actor"])


def test_replay_to_learner_roundtrip(eng_mod):
    """sample -> iteration -> priority write-back on device, no host round trip of the batch."""
    cfg = eng_mod.PathConfig(obs=6, act=2, hidden=64, batch=16, burn_in=5, learning=8, n_step=3)
    rng = np.random.default_rng(2)
    rp = eng_mod.DeviceReplay(cfg, capacity_rows=20000)
    for _ in range(40):
        E = int(rng.integers(40, 200))
        n_rows = E + cfg.n_step
        term = np.zeros(n_rows, np.float32)
        term[E:] = 1
        rp.add_episode(rng.standard_normal((n_rows, 6)).astype(np.float32), rng.uniform(-1, 1, (n_rows, 2)).astype(np.float32),
                       rng.standard_normal(n_rows).astype(np.float32), term,
                       (0.1 * rng.standard_normal((E, 4, 2, 64))).astype(np.float32),
                       rng.uniform(0.01, 1, E - 13).astype(np.float32))
    eng = eng_mod.LearnerEngine(cfg)
    gen = torch.Generator(device="cuda").manual_seed(0)
    for _ in range(3):
        rp.sample_into(eng, generator=gen)
        eng.step()
        rp.update_priorities(eng.leaf_idx, eng.priority)
    torch.cuda.synchronize()
    leaves = rp.tree_level(0)
    li = eng.leaf_idx.cpu().numpy()
    pr = eng.priority.cpu().numpy()
    last = {int(l): float(p) for l, p in zip(li, pr)}
    for l, p in last.items():
        assert leaves[l].item() == np.float32(p)
    assert np.isfinite(pr).all() and (pr >= 0).all()


EDGE_CASES = [
    # obs, act, hidden, batch, burn_in, learning, n_step  (same list as tests/test_oracle_golden.py)
    (3, 1, 32, 1, 1, 2, 1),
    (5, 2, 32, 3, 1, 3, 2),
    (4, 3, 64, 5, 2, 6, 4),
    (6, 2, 96, 2, 3, 4, 5),
]


@pytest.mark.parametrize("obs,act,hidden,batch,burn_in,learning,n_step", EDGE_CASES)
def test_edge_shapes_against_port(eng_mod, obs, act, hidden, batch, burn_in, learning, n_step):
    """B = 1, A = 1, n_step = 1, minimal burn-in, a hidden size on the generic scan path: two consecutive iterations
    against the CPU port (which tests/test_oracle_golden.py pins to the unmodified reference)."""
    pc = ref_port.PathConfig(obs=obs, act=act, hidden=hidden, batch=batch, burn_in=burn_in, learning=learning, n_step=n_step)
    torch.set_num_threads(1)
    port = ref_port.PortLearner(pc, seed=11)
    cfg = eng_mod.PathConfig(obs=obs, act=act, hidden=hidden, batch=batch, burn_in=burn_in, learning=learning, n_step=n_step)
    eng = eng_mod.LearnerEngine(cfg)
    sd = lambda m: {k: v.detach().numpy() for k, v in m.state_dict().items()}  # noqa: E731
    eng.load_state_dicts(sd(port.actor), sd(port.critic))
    for it in range(2):
        batch_np = ref_port.synthetic_batch(pc, seed=100 + it)
        ref = port.iteration(batch_np)
        eng.set_batch(batch_np)
        eng.step()
        torch.cuda.synchronize()
        errs = {"q": rel_l2(eng.q_value.cpu().numpy(), ref["q_value"]),
                "target": rel_l2(eng.target_q_value.cpu().numpy(), ref["target_q_value"]),
                "prio": rel_l2(eng.priority.cpu().numpy(), ref["priority"])}
        for net in ("actor", "critic"):
            gr, pa = flat_sd(eng.views(net, "grads")), flat_sd(eng.views(net))
            for k in eng_mod.PARAM_KEYS:
                errs[f"{net}_grad/{k}"] = rel_l2(gr[k], ref[f"{net}_grad"][k])
                errs[f"{net}_after/{k}"] = rel_l2(pa[k], ref[f"{net}_after"][k])
        bad = {k: v for k, v in errs.items() if not v < TOL}
        assert not bad, f"iteration {it}: {bad}"


def test_training_state_resume_continues_the_run(eng_mod):
    """Next-row N3: nets + Adam moments + step counter round-trip; an engine restored from the state after 2 iterations
    continues like the one that never stopped (Adam bias correction and the target period depend on the step; the
    comparison allows for the run-to-run rounding of the split-K reductions, nothing more)."""
    pc = ref_port.PathConfig(obs=6, act=2, hidden=64, batch=8, burn_in=4, learning=6, n_step=2, target_interval=3)
    cfg = eng_mod.PathConfig(obs=6, act=2, hidden=64, batch=8, burn_in=4, learning=6, n_step=2, target_interval=3)
    a = eng_mod.LearnerEngine(cfg, seed=9)
    for it in range(2):
        a.set_batch(ref_port.synthetic_batch(pc, seed=it))
        a.step()
    st = a.training_state()
    assert st["step"] == 2 and set(st) >= {"actor", "critic", "target_actor", "target_critic", "actor_optimizer", "critic_optimizer"}
    b = eng_mod.LearnerEngine(cfg, seed=123)          # different initial weights: everything must come from the state
    b.load_training_state(st)
    assert b.step_count == 2
    for it in range(2, 5):                             # crosses a hard target update (step 3)
        batch = ref_port.synthetic_batch(pc, seed=it)
        for e in (a, b):
            e.set_batch(batch)
            e.step()
    torch.cuda.synchronize()
    for net in ("actor", "critic", "target_actor", "target_critic"):
        assert rel_l2(a.flat[net].cpu().numpy(), b.flat[net].cpu().numpy()) < 1e-5, net
    for net in ("actor", "critic"):
        assert rel_l2(a.exp_avg[net].cpu().numpy(), b.exp_avg[net].cpu().numpy()) < 1e-4
        assert rel_l2(a.exp_avg_sq[net].cpu().numpy(), b.exp_avg_sq[net].cpu().numpy()) < 1e-4
    assert torch.equal(a.flat["target_critic"], a.flat["critic"]) == torch.equal(b.flat["target_critic"], b.flat["critic"])


@pytest.mark.parametrize("hidden,batch", [(64, 8), (128, 32)])
def test_pipelined_step_matches_sequential(eng_mod, hidden, batch):
    """`step(prefetch=...)`: the next batch is drawn mid-iteration into the second batch slot and its target chains run
    before the actor phase of the iteration in flight (r2d2_learner_target_phase); on iterations that copy into the
    target nets the hook is called at the end instead.  Same batches in the same order must give the same run as the
    sequential sample -> step -> write-back loop, including the priorities handed to the hook."""
    kw = dict(obs=6, act=2, hidden=hidden, batch=batch, burn_in=4, learning=6, n_step=2, target_interval=3)
    pc = ref_port.PathConfig(**kw)
    cfg = eng_mod.PathConfig(**kw)
    steps = 8                                               # crosses two hard target updates
    batches = [ref_port.synthetic_batch(pc, seed=40 + it) for it in range(steps + 1)]
    seq = eng_mod.LearnerEngine(cfg, seed=3)
    seq_prio = []
    for it in range(steps):
        seq.set_batch(batches[it])
        seq.step()
        seq_prio.append(seq.priority.clone())
    pip = eng_mod.LearnerEngine(cfg, seed=3)
    pip_prio, calls = [], []
    pip.set_batch(batches[0])
    for it in range(steps):
        def hook(eng, used, it=it):
            calls.append(it)
            pip_prio.append(used.priority.clone())
            eng.set_batch(batches[it + 1])
        pip.step(prefetch=hook)
    torch.cuda.synchronize()
    assert calls == list(range(steps))
    assert pip.step_count == seq.step_count == steps
    for it in range(steps):
        assert rel_l2(pip_prio[it].cpu().numpy(), seq_prio[it].cpu().numpy()) < 1e-5, it
    for net in ("actor", "critic", "target_actor", "target_critic"):
        assert rel_l2(pip.flat[net].cpu().numpy(), seq.flat[net].cpu().numpy()) < 1e-5, net
    assert pip.launches_per_iteration == seq.launches_per_iteration
    with pytest.raises(Exception, match="target chains"):       # the prefetched batch is final until the next step
        pip.set_batch(batches[0])
    pip.discard_prefetched()
    for e in (seq, pip):                                        # ... or explicitly dropped: both engines continue alike
        e.set_batch(batches[1])
        e.step()
    torch.cuda.synchronize()
    for net in ("actor", "critic"):
        assert rel_l2(pip.flat[net].cpu().numpy(), seq.flat[net].cpu().numpy()) < 1e-5, net
