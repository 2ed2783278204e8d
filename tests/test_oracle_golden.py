"""Pin the oracles (oracle/ref_port.py, oracle/learner_oracle.py) against fixtures produced by
the UNMODIFIED reference (oracle/make_golden.py).  CPU only."""
import numpy as np
import pytest
import torch

from conftest import checked_state, golden_batch, golden_cfg, golden_init, golden_sample, load_golden, rel_l2
from oracle import learner_oracle as lo
from oracle import ref_port

CASES = [("ref_walker_h128.npz", 1), ("ref_pend_h128.npz", 2), ("ref_tiny_h32.npz", 4)]


@pytest.mark.parametrize("name,seed", CASES)
def test_port_init_bit_identical(name, seed):
    """Same torch seed -> the port's nets equal the reference's models.py nets bit for bit."""
    g = load_golden(name)
    lr = ref_port.PortLearner(golden_cfg(g), seed=seed)
    for net, mod in (("actor", lr.actor), ("critic", lr.critic)):
        checked_state(g, f"init_sha256/{net}", mod)


@pytest.mark.parametrize("name,seed", CASES)
def test_port_iterations_match_reference(name, seed):
    g = load_golden(name)
    torch.set_num_threads(4)
    lr = ref_port.PortLearner(golden_cfg(g))
    lr.load_params(*golden_init(g))
    for it in range(int(g["n_iters"])):
        out = lr.iteration(golden_batch(g, it))
        assert rel_l2(out["q_value"], g[f"it{it}/q_value"]) < 2e-6
        assert rel_l2(out["target_q_value"], g[f"it{it}/target_q_value"]) < 2e-6
        assert abs(out["critic_loss"] - float(g[f"it{it}/critic_loss"])) <= 1e-6 * abs(float(g[f"it{it}/critic_loss"]))
        assert abs(out["actor_loss"] - float(g[f"it{it}/actor_loss"])) <= 1e-5 * abs(float(g[f"it{it}/actor_loss"])) + 1e-9
        assert rel_l2(out["priority"], g[f"it{it}/priority_written"]) < 1e-6
        for net in ("actor", "critic"):
            for k in ref_port.PARAM_KEYS:
                assert abs(np.linalg.norm(out[f"{net}_grad"][k].astype(np.float64)) -
                           float(g[f"it{it}/{net}_grad_norm/{k}"])) <= 2e-4 * float(g[f"it{it}/{net}_grad_norm/{k}"]) + 1e-12
                assert rel_l2(out[f"{net}_after"][k].reshape(-1)[::97], g[f"it{it}/{net}_after_sub/{k}"]) < 1e-5
        if it == 0:
            for net in ("actor", "critic"):
                for k in ref_port.PARAM_KEYS:
                    assert rel_l2(golden_sample(g, 0, net, k, out[f"{net}_grad"][k]), g[f"it0/{net}_grad/{k}"]) < 1e-4, (net, k)
                    assert rel_l2(golden_sample(g, 0, net, k, out[f"{net}_after"][k]), g[f"it0/{net}_after/{k}"]) < 1e-6, (net, k)


@pytest.mark.parametrize("name,seed", CASES)
def test_numpy_oracle_matches_reference(name, seed):
    """float64 manual-BPTT oracle vs the reference's fp32 autograd: agreement at fp32 round-off."""
    g = load_golden(name)
    c = golden_cfg(g)
    init = dict(zip(("actor", "critic"), golden_init(g)))
    ol = lo.OracleLearner(init["actor"], init["critic"], burn_in=c.burn_in, learning=c.learning, n_step=c.n_step)
    for it in range(int(g["n_iters"])):
        out = ol.iteration(golden_batch(g, it))
        assert rel_l2(out["q_value"], g[f"it{it}/q_value"]) < 5e-5
        assert rel_l2(out["target_q_value"], g[f"it{it}/target_q_value"]) < 5e-5
        assert abs(out["critic_loss"] - float(g[f"it{it}/critic_loss"])) < 1e-5 * abs(float(g[f"it{it}/critic_loss"]))
        assert abs(out["actor_loss"] - float(g[f"it{it}/actor_loss"])) < 1e-4 * abs(float(g[f"it{it}/actor_loss"])) + 1e-8
        assert rel_l2(out["priority"], g[f"it{it}/priority_written"]) < 5e-5
        assert rel_l2(out["average_td_loss"], g[f"it{it}/average_td_loss"]) < 5e-5
        if it == 0:
            for net in ("actor", "critic"):
                for k in lo.PARAM_KEYS:
                    assert rel_l2(golden_sample(g, 0, net, k, out[f"{net}_grad"][k]), g[f"it0/{net}_grad/{k}"]) < 2e-4, (net, k)
                    # Adam's first step is sign-like (|update| = lr); compare the update, not the params
                    init0 = golden_sample(g, 0, net, k, init[net][k])
                    upd = golden_sample(g, 0, net, k, out[f"{net}_after"][k]) - init0
                    ref_upd = g[f"it0/{net}_after/{k}"].astype(np.float64) - init0
                    assert rel_l2(upd, ref_upd) < 5e-2, (net, k)
        for net in ("actor", "critic"):
            for k in lo.PARAM_KEYS:
                assert rel_l2(out[f"{net}_after"][k].reshape(-1)[::97], g[f"it{it}/{net}_after_sub/{k}"]) < 2e-4


def test_known_answers():
    k = load_golden("ref_kat.npz")
    assert abs(ref_port.sequence_priority(k["calc_priority_in"]) - float(k["calc_priority_out"])) < 1e-6
    assert abs(float(k["calc_priority_out"]) - 3.85) < 1e-6
    assert np.allclose(ref_port.value_rescale(torch.tensor(k["h_in"])).numpy(), k["h_out"], rtol=1e-6, atol=0)
    assert np.allclose(lo.value_rescale(k["h_in"].astype(np.float64)), k["h_out"], rtol=1e-5, atol=1e-7)
    assert np.allclose(k["h_out"][:4], [-1, 0, 1, 2])
    assert list(k["slice_b4"]) == [3, 3, 3, 2]          # learner.py:137 drops the last step of b = B-1
    for row, want in zip(k["prio_in"], k["prio_out"]):
        assert abs(ref_port.sequence_priority(row) - want) < 1e-6


EDGE_CASES = [
    # obs, act, hidden, batch, burn_in, learning, n_step  - shapes the goldens do not reach
    (3, 1, 32, 1, 1, 2, 1),      # single sequence, single action, n_step 1: the [b:-1:B] slice drops the ONLY last row
    (5, 2, 32, 3, 1, 3, 2),      # shortest burn-in the reference supports (learner.py:93-95 needs >= 1 row)
    (4, 3, 64, 5, 2, 6, 4),      # n_step close to the learning length
    (6, 2, 96, 2, 3, 4, 5),      # hidden size outside the cluster kernels (generic scan path on the GPU)
]


@pytest.mark.parametrize("obs,act,hidden,batch,burn_in,learning,n_step", EDGE_CASES)
def test_numpy_oracle_matches_port_on_edge_shapes(obs, act, hidden, batch, burn_in, learning, n_step):
    """The float64 manual-BPTT restatement (the per-kernel parity target of the CUDA tests) against the torch port
    (autograd, pinned to the unmodified reference by the tests above) where the reference goldens have no fixture:
    B = 1, A = 1, n_step = 1, minimal burn-in, odd hidden sizes.  Two consecutive iterations (Adam state carried)."""
    torch.set_num_threads(1)
    pc = ref_port.PathConfig(obs=obs, act=act, hidden=hidden, batch=batch, burn_in=burn_in, learning=learning, n_step=n_step)
    port = ref_port.PortLearner(pc, seed=11)
    sd = lambda m: {k: v.detach().numpy().copy() for k, v in m.state_dict().items()}  # noqa: E731
    ol = lo.OracleLearner(sd(port.actor), sd(port.critic), burn_in=burn_in, learning=learning, n_step=n_step)
    for it in range(2):
        batch_np = ref_port.synthetic_batch(pc, seed=100 + it)
        ref = port.iteration(batch_np)
        out = ol.iteration(batch_np)
        assert rel_l2(out["q_value"], ref["q_value"]) < 5e-5
        assert rel_l2(out["target_q_value"], ref["target_q_value"]) < 5e-5
        assert rel_l2(out["priority"], ref["priority"]) < 5e-5
        assert abs(out["critic_loss"] - ref["critic_loss"]) < 1e-4 * abs(ref["critic_loss"]) + 1e-9
        assert abs(out["actor_loss"] - ref["actor_loss"]) < 1e-4 * abs(ref["actor_loss"]) + 1e-9
        for net in ("actor", "critic"):
            for k in lo.PARAM_KEYS:
                assert rel_l2(out[f"{net}_grad"][k], ref[f"{net}_grad"][k]) < 5e-4, (it, net, k)
