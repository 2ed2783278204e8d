import functools
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "pytorch-r2d2-dpg_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if has_gpu:
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


def load_golden(name):
    z = np.load(os.path.join(GOLDEN, name), allow_pickle=False)
    return {k: z[k] for k in z.files}


def checked_state(g, prefix, net):
    """state dict of a port net as numpy, asserted bit-identical to the reference net whose digests the fixture
    stores under 'prefix/<key>'."""
    from oracle.make_golden import array_digest
    sd = {k: v.detach().numpy().copy() for k, v in net.state_dict().items()}
    for k, v in sd.items():
        assert array_digest(v) == str(g[f"{prefix}/{k}"]), (prefix, k)
    return sd


def golden_cfg(g):
    from oracle import ref_port
    return ref_port.PathConfig(obs=int(g["cfg/obs_size"]), act=int(g["cfg/n_actions"]), hidden=int(g["cfg/hidden"]),
                               batch=int(g["cfg/batch_size"]), burn_in=int(g["cfg/burn_in"]),
                               learning=int(g["cfg/learning"]), n_step=int(g["cfg/n_step"]))


def golden_init(g):
    """(actor, critic) initial weights of the reference learner: the port's nets under the same torch seed."""
    from oracle import ref_port
    lr = ref_port.PortLearner(golden_cfg(g), seed=int(g["cfg/seed"]))
    return checked_state(g, "init_sha256/actor", lr.actor), checked_state(g, "init_sha256/critic", lr.critic)


@functools.lru_cache(maxsize=4)
def _golden_replay(obs, act, hidden, burn_in, learning, n_step, n_episodes, episode_len, data_seed):
    from oracle import ref_port
    cfg = ref_port.PathConfig(obs=obs, act=act, hidden=hidden, burn_in=burn_in, learning=learning, n_step=n_step)
    f = ref_port.synthetic_actor_file(obs_size=obs, n_actions=act, hidden=hidden, n_episodes=n_episodes,
                                      episode_len=episode_len, seed=data_seed, burn_in=burn_in, learning=learning,
                                      n_step=n_step)
    rp = ref_port.PortReplay(cfg)
    for rows, states, prio in zip(f["replay_memory"], f["recurrent_state"], f["priority"]):
        rp.add_episode(rows, states, prio)
    return rp


def golden_batch(g, it):
    """Batch the reference sampled in iteration `it`: its (episode, sequence) draws gathered from the synthetic actor
    file it learned from, asserted bit-identical to the digests of the batch it trained on."""
    from oracle.make_golden import BATCH_KEYS, array_digest
    rp = _golden_replay(*(int(g[f"cfg/{k}"]) for k in ("obs_size", "n_actions", "hidden", "burn_in", "learning",
                                                       "n_step", "n_episodes", "episode_len", "data_seed")))
    batch = rp.gather([int(e) for e in g[f"it{it}/episode_index"]], [int(s) for s in g[f"it{it}/sequence_index"]])
    batch = {k: batch[k].numpy() for k in BATCH_KEYS}
    for k, v in batch.items():
        assert array_digest(v) == str(g[f"it{it}/sha256/{k}"]), (it, k)
    return batch


def golden_sample(g, it, net, k, a):
    """The elements of a full tensor `a` that the fixture keeps of the reference's '<net>_grad' / '<net>_after'."""
    return np.asarray(a).reshape(-1)[g[f"it{it}/sample_idx/{net}/{k}"]]


def rel_l2(a, b):
    a = np.asarray(a, np.float64).ravel()
    b = np.asarray(b, np.float64).ravel()
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))
