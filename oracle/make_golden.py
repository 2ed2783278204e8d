"""Generate tests/golden/*.npz by executing the UNMODIFIED reference (/root/reference) on CPU.

Run in the build container only (the reference is not present on the GPU box):
    python oracle/make_golden.py
The fixtures pin the oracles (oracle/ref_port.py, oracle/learner_oracle.py) and, through them,
the CUDA path.  torch version used is recorded in each file (the reference pins none).

Files
  ref_walker_h128.npz   real learner.py + real models.py, walker/run sizes O=24 A=6 H=128 B=32
                        Bn=20 L=40 n=5 (the reference as-is, learner.py:29-34), 3 iterations
  ref_pend_h128.npz     same code, Pendulum shape O=3 A=1, B=8, 2 iterations (A=1 edge case)
  ref_tiny_h32.npz      real learner.py driving the hidden-parameterised nets (oracle/ref_port.py
                        make_models_module) O=5 A=2 H=32 B=4 Bn=6 L=10 n=3, 3 iterations
  ref_kat.npz           known answers of utils.calc_priority / utils.invertical_vf and the
                        priority slice rule (SURVEY section 4)
  ref_sampler_hist.npz  empirical (episode, sequence) histogram of the real two-level sampler
                        (replay_memory.py:95-114) on a small memory, for the chi-square test
  ref_ingest.npz        the real LearnerReplayMemory.load (replay_memory.py:138-157) over a deterministic sequence of actor
                        files with a small sequence cap: sequence_counter and surviving episodes after every file
  ref_actor_prio.npz    the real Actor.calc_nstep_reward / Actor.calc_priorities (actor.py:74-107) on synthetic
                        episodes of several lengths: raw and n-step rewards, torch seed and weight digests of
                        the three nets the pass reads, and the initial priorities it produced (next-row N2 of
                        SURVEY 8f)
Inputs that the tests can rebuild - initial weights from the torch seed with the oracle/ref_port.py nets, sampled
batches from the synthetic actor file and the drawn (episode, sequence) indices - are stored as SHA-256 digests
(array_digest), and the rebuilt arrays are checked against them bit for bit.
"""
from __future__ import annotations

import hashlib
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import ref_harness, ref_port  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
NETS = ("actor", "critic")
BATCH_KEYS = ("obs", "act", "rew", "term", "a_state", "ta_state", "c_state", "tc_state")
SAMPLE = 4096          # elements kept of a full gradient / weight tensor of the iterations in `full_iters`


def array_digest(a) -> str:
    """SHA-256 of dtype, shape and bytes: lets a fixture pin an input that the tests rebuild (initial weights from
    the torch seed, sampled batches from the synthetic actor file) bit for bit without storing it."""
    a = np.ascontiguousarray(a)
    return hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).hexdigest()


def _sample_index(n):
    """Sorted, seeded sample of SAMPLE flat positions (all of them for a smaller tensor), stored with the values."""
    if n <= SAMPLE:
        return np.arange(n, dtype=np.int32)
    return np.sort(np.random.default_rng(n).choice(n, SAMPLE, replace=False)).astype(np.int32)


def _flatten(records, full_iters=(0,)):
    """Everything the reference computed, with its inputs (initial weights, batches) as digests and the full
    gradient / weight tensors of `full_iters` as a fixed sample: every fixture stays under 1 MB."""
    out = {"n_iters": np.int64(len(records)), "torch_version": np.array(torch.__version__)}
    r0 = records[0]
    for net in NETS:
        for k, v in r0[f"{net}_init"].items():
            out[f"init_sha256/{net}/{k}"] = np.array(array_digest(v))
    for i, r in enumerate(records):
        for k in BATCH_KEYS:
            out[f"it{i}/sha256/{k}"] = np.array(array_digest(r[k]))
        for k in ("episode_index", "sequence_index", "q_value", "target_q_value", "critic_loss",
                  "actor_loss", "average_td_loss", "priority_written", "total_priority_written"):
            out[f"it{i}/{k}"] = np.asarray(r[k])
        for net in NETS:
            for k, v in r[f"{net}_grad"].items():
                if i in full_iters:
                    idx = _sample_index(v.size)
                    out[f"it{i}/sample_idx/{net}/{k}"] = idx
                    out[f"it{i}/{net}_grad/{k}"] = v.reshape(-1)[idx]
                out[f"it{i}/{net}_grad_norm/{k}"] = np.float64(np.linalg.norm(v.astype(np.float64)))
            for k, v in r[f"{net}_after"].items():
                if i in full_iters:
                    out[f"it{i}/{net}_after/{k}"] = v.reshape(-1)[out[f"it{i}/sample_idx/{net}/{k}"]]
                out[f"it{i}/{net}_after_norm/{k}"] = np.float64(np.linalg.norm(v.astype(np.float64)))
                out[f"it{i}/{net}_after_sub/{k}"] = v.reshape(-1)[::97].copy()
    return out


def gen_learner(name, models_module=None, **kw):
    recs, times, lr = ref_harness.run_reference_learner(models_module=models_module, **kw)
    d = _flatten(recs)
    d["config"] = np.array(repr(kw))
    for k in ("obs_size", "n_actions", "hidden", "batch_size", "burn_in", "learning", "n_step", "seed", "data_seed",
              "episode_len"):
        d[f"cfg/{k}"] = np.int64(kw.get(k, {"hidden": 128, "batch_size": 32, "burn_in": 20,
                                          "learning": 40, "n_step": 5, "episode_len": 250}.get(k, 0)))
    d["cfg/n_episodes"] = np.int64(len(lr.memory.memory))      # the one actor file the batches were drawn from
    path = os.path.join(OUT, name)
    np.savez_compressed(path, **d)
    print(name, "iters", len(recs), "iter-times", np.round(times, 3), "size %.2f MB" % (os.path.getsize(path) / 1e6))


def gen_kat():
    sys.path.insert(0, ref_harness.REFERENCE_DIR)
    for m in ("utils",):
        sys.modules.pop(m, None)
    import utils as ref_utils
    d = {
        "calc_priority_in": np.float32([1, 2, 3, 4]),
        "calc_priority_out": np.float64(ref_utils.calc_priority(np.float32([1, 2, 3, 4]))),
        "h_in": np.float32([-3, 0, 3, 8, -0.5, 1e-3, 100.0, -1e4]),
    }
    d["h_out"] = ref_utils.invertical_vf(torch.tensor(d["h_in"])).numpy()
    d["slice_b4"] = np.array([len(np.arange(12)[i:-1:4]) for i in range(4)])
    rng = np.random.default_rng(3)
    td = rng.uniform(0, 2, (7, 40)).astype(np.float32)
    d["prio_in"] = td
    d["prio_out"] = np.array([ref_utils.calc_priority(r) for r in td], dtype=np.float64)
    np.savez_compressed(os.path.join(OUT, "ref_kat.npz"), **d)
    sys.modules.pop("utils", None)
    sys.path.remove(ref_harness.REFERENCE_DIR)
    print("ref_kat.npz ok")


def gen_sampler_hist(n_draw_batches=400, batch=32):
    """Real LearnerReplayMemory.sample() index stream histogram (replay_memory.py:99-119)."""
    ref_harness._install_stubs(3, 1)
    torch.Tensor.cuda = lambda self, *a, **k: self
    sys.path.insert(0, ref_harness.REFERENCE_DIR)
    for m in ("replay_memory",):
        sys.modules.pop(m, None)
    import replay_memory as ref_rm
    rng = np.random.default_rng(11)
    mem = ref_rm.LearnerReplayMemory(memory_sequence_size=10 ** 6, batch_size=batch)
    ep_lens = [70, 90, 66, 120, 75]
    prios = []
    for E in ep_lens:
        rows = [(np.zeros(3, np.float32), np.zeros(1, np.float32), [0.0], [0.0]) for _ in range(E + 5)]
        st = [[[np.zeros(4, np.float32), np.zeros(4, np.float32)] for _ in range(4)] for _ in range(E)]
        p = [float(np.float32(rng.uniform(0.01, 1.0))) for _ in range(E - 60)]
        mem.memory.append(rows)
        mem.recurrent_state.append(st)
        mem.priority.append(p)
        mem.total_priority.append(sum(p))
        prios.append(np.asarray(p, np.float64))
    torch.manual_seed(5)
    offs = np.concatenate([[0], np.cumsum([len(p) for p in prios])])
    counts = np.zeros(offs[-1], np.int64)
    for _ in range(n_draw_batches):
        out = mem.sample()
        for e, s in zip(out[0], out[1]):
            counts[offs[e] + s] += 1
    np.savez_compressed(os.path.join(OUT, "ref_sampler_hist.npz"), counts=counts,
                        priorities=np.concatenate(prios), episode_offsets=offs,
                        n_draws=np.int64(n_draw_batches * batch))
    sys.modules.pop("replay_memory", None)
    sys.path.remove(ref_harness.REFERENCE_DIR)
    print("ref_sampler_hist.npz ok", counts.sum())


def ingest_file_sequence(seed=21, n_files=6, obs_size=4, n_actions=2, hidden=8):
    """Deterministic sequence of actor files (each: list of episodes in the reference's tuple format) used by the ingest
    parity fixture and regenerated, from the same seed, by tests/test_gpu_replay.py."""
    rng = np.random.default_rng(seed)
    files = []
    tag = 0
    for f in range(n_files):
        eps = []
        for _ in range(int(rng.integers(2, 5))):
            E = int(rng.integers(60, 140))
            tag += 1
            rows = [(np.full(obs_size, tag + 0.001 * t, np.float32), rng.uniform(-1, 1, n_actions).astype(np.float32),
                     [float(rng.standard_normal())], [0.0]) for t in range(E)]
            rows += [(np.zeros(obs_size, np.float32), np.zeros(n_actions, np.float32), [0.0], [1.0]) for _ in range(5)]
            st = [[[rng.standard_normal(hidden).astype(np.float32) * 0.1, rng.standard_normal(hidden).astype(np.float32) * 0.1]
                   for _ in range(4)] for _ in range(E)]
            pr = [float(np.float32(rng.uniform(0.01, 1.0))) for _ in range(E - 60)]
            eps.append((rows, st, pr, tag))
        files.append((f % 3, eps))                            # three actors write in turn
    return files


def gen_ingest():
    """The real LearnerReplayMemory.load (replay_memory.py:138-157) over the file sequence above with a small
    memory_sequence_size so that the FIFO eviction and its asymmetric counter (:147 vs :149) are exercised."""
    import tempfile
    from collections import deque
    ref_harness._install_stubs(4, 2)
    torch.Tensor.cuda = lambda self, *a, **k: self
    if not getattr(torch.load, "_r2d2_patched", False):
        _orig = torch.load

        def _load(*a, **k):
            k.setdefault("weights_only", False)
            return _orig(*a, **k)
        _load._r2d2_patched = True
        torch.load = _load
    if ref_harness.REFERENCE_DIR not in sys.path:
        sys.path.insert(0, ref_harness.REFERENCE_DIR)
    sys.modules.pop("replay_memory", None)
    import replay_memory as ref_rm
    cwd = os.getcwd()
    os.chdir(tempfile.mkdtemp(prefix="r2d2_ingest_"))
    os.makedirs("memory_data")
    try:
        cap = 150
        mem = ref_rm.LearnerReplayMemory(memory_sequence_size=cap, batch_size=4)
        counters, survivors = [], []
        for actor_id, eps in ingest_file_sequence():
            torch.save({"replay_memory": deque([e[0] for e in eps]), "recurrent_state": deque([e[1] for e in eps]),
                        "priority": deque([e[2] for e in eps]), "total_priority": [sum(e[2]) for e in eps]},
                       "memory_data/memory{}.pt".format(actor_id))
            mem.load(actor_id)
            counters.append(mem.sequence_counter)
            survivors.append([int(round(float(ep[0][0][0]))) for ep in mem.memory])   # the tag in obs[0] of the first row
            assert len(torch.load("memory_data/memory{}.pt".format(actor_id))["replay_memory"]) == 0   # handed back emptied
    finally:
        os.chdir(cwd)
        sys.modules.pop("replay_memory", None)
    d = {"memory_sequence_size": np.int64(cap), "sequence_counter": np.int64(counters),
         "n_files": np.int64(len(counters))}
    for i, sv in enumerate(survivors):
        d[f"survivors/{i}"] = np.int64(sv)
    np.savez_compressed(os.path.join(OUT, "ref_ingest.npz"), **d)
    print("ref_ingest.npz ok", counters, [len(x) for x in survivors])


def gen_actor_priorities():
    """Real Actor.calc_nstep_reward + Actor.calc_priorities (actor.py:74-107), incl. the deque-of-40 off-by-one
    (window of priority k covers TD steps k+21..k+60) and the mean-then-square TD (not the learner's squared mean)."""
    d = {"torch_version": np.array(torch.__version__)}
    cases = [("walker", 24, 6, [61, 75, 130]), ("pend", 3, 1, [60, 64, 97])]
    d["n_cases"] = np.int64(len(cases))
    for ci, (name, O, A, lens) in enumerate(cases):
        ref_harness._install_stubs(O, A)
        ident = lambda self, *a, **k: self  # noqa: E731
        torch.Tensor.cuda = ident
        torch.nn.Module.cuda = ident
        for m in ("actor", "replay_memory", "models", "utils", "learner"):
            sys.modules.pop(m, None)
        if ref_harness.REFERENCE_DIR not in sys.path:
            sys.path.insert(0, ref_harness.REFERENCE_DIR)
        import tempfile
        cwd = os.getcwd()
        os.chdir(tempfile.mkdtemp(prefix="r2d2_actor_"))     # no model_data/model.pt: load_model() is a no-op (actor.py:51)
        try:
            import actor as ref_actor
            import models as ref_models
            torch.manual_seed(100 + ci)
            a = ref_actor.Actor(0)
            # the constructor deep-copies the online nets into the targets (actor.py:43-45): give the targets their own
            # weights so that the fixture distinguishes the four roles
            a.target_actor = ref_models.ActorNet(O, A, 0).eval()
            a.target_critic = ref_models.CriticNet(O, A, 0).eval()
            d[f"c{ci}/seed"] = np.int64(100 + ci)
            for net_name in ("critic", "target_actor", "target_critic"):
                for k, v in getattr(a, net_name).state_dict().items():
                    d[f"c{ci}/{net_name}/{k}"] = np.array(array_digest(v.detach().numpy()))
            d[f"c{ci}/cfg"] = np.int64([O, A, 128, a.burn_in_length, a.learning_length, a.n_step])
            d[f"c{ci}/gamma"] = np.float64(a.gamma)
            d[f"c{ci}/n_episodes"] = np.int64(len(lens))
            rng = np.random.default_rng(40 + ci)
            for ei, E in enumerate(lens):
                seq = [(rng.standard_normal(O).astype(np.float32), rng.uniform(-1, 1, A).astype(np.float32),
                        [float(rng.standard_normal())], [0.0]) for _ in range(E)]
                seq[-1][3][0] = 1.0                                                   # time_step.last() on the final real row
                seq += [(np.zeros(O, np.float32), np.zeros(A, np.float32), [0.0], [1.0]) for _ in range(a.n_step)]  # actor.py:173
                raw = np.asarray([r[2][0] for r in seq], np.float64)
                a.sequence = seq
                a.calc_nstep_reward()
                with torch.no_grad():
                    a.calc_priorities()
                d[f"c{ci}/e{ei}/obs"] = np.stack([r[0] for r in seq])
                d[f"c{ci}/e{ei}/act"] = np.stack([r[1] for r in seq])
                d[f"c{ci}/e{ei}/rew_raw"] = raw
                d[f"c{ci}/e{ei}/rew_nstep"] = np.asarray([r[2][0] for r in seq], np.float64)
                d[f"c{ci}/e{ei}/term"] = np.asarray([r[3][0] for r in seq], np.float32)
                d[f"c{ci}/e{ei}/priority"] = np.asarray(a.priority, np.float64)
                assert len(a.priority) == E - a.sequence_length
        finally:
            os.chdir(cwd)
            for m in ("actor", "replay_memory", "models", "utils"):
                sys.modules.pop(m, None)
    np.savez_compressed(os.path.join(OUT, "ref_actor_prio.npz"), **d)
    print("ref_actor_prio.npz ok")


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(8)
    if len(sys.argv) > 1 and sys.argv[1] == "actor":
        gen_actor_priorities()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "ingest":
        gen_ingest()
        sys.exit(0)
    gen_kat()
    gen_actor_priorities()
    gen_ingest()
    gen_sampler_hist()
    gen_learner("ref_walker_h128.npz", obs_size=24, n_actions=6, n_iters=3, seed=1, data_seed=0)
    gen_learner("ref_pend_h128.npz", obs_size=3, n_actions=1, batch_size=8, n_iters=2, seed=2, data_seed=3)
    gen_learner("ref_tiny_h32.npz", models_module=ref_port.make_models_module(32), obs_size=5,
                n_actions=2, hidden=32, batch_size=4, burn_in=6, learning=10, n_step=3, n_iters=3,
                seed=4, data_seed=5, episode_len=60)
