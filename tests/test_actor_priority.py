"""Next-row N2 (SURVEY 8f): actor-side n-step reward pre-sum and initial priorities (/root/reference/actor.py:74-107).

 * CPU: the numpy restatement (oracle/actor_oracle.py) against the fixture the UNMODIFIED reference produced
   (tests/golden/ref_actor_prio.npz, oracle/make_golden.py gen_actor_priorities) - pins the checker;
 * GPU: the batched device pass (r2d2_b200.actor_priority: three persistent chains + r2d2_actor_priorities,
   r2d2_nstep_rewards) against the same fixture, 1e-3 relative (north_star tolerance)."""
import numpy as np
import pytest

from conftest import checked_state, load_golden, rel_l2

def _nets(g, ci, O, A, H):
    """The three nets the reference's pass read: under its torch seed the actor builds actor, critic, then the fixture
    target actor, target critic (oracle/make_golden.py gen_actor_priorities); the port's nets draw the same weights."""
    import torch
    from oracle import ref_port
    torch.manual_seed(int(g[f"c{ci}/seed"]))
    ref_port.PortActorNet(O, A, 0, H)
    made = {"critic": ref_port.PortCriticNet(O, A, 0, H), "target_actor": ref_port.PortActorNet(O, A, 0, H),
            "target_critic": ref_port.PortCriticNet(O, A, 0, H)}
    return {net: checked_state(g, f"c{ci}/{net}", m) for net, m in made.items()}


def _case(g, ci):
    O, A, H, Bn, L, n = (int(x) for x in g[f"c{ci}/cfg"])
    nets = _nets(g, ci, O, A, H)
    eps = []
    for ei in range(int(g[f"c{ci}/n_episodes"])):
        eps.append({k: g[f"c{ci}/e{ei}/{k}"] for k in ("obs", "act", "rew_raw", "rew_nstep", "term", "priority")})
    return (O, A, H, Bn, L, n, float(g[f"c{ci}/gamma"])), nets, eps


def test_actor_oracle_matches_reference_fixture():
    from oracle import actor_oracle as ao
    g = load_golden("ref_actor_prio.npz")
    for ci in range(int(g["n_cases"])):
        (O, A, H, Bn, L, n, gamma), nets, eps = _case(g, ci)
        for e in eps:
            assert np.allclose(ao.nstep_rewards(e["rew_raw"], n, gamma), e["rew_nstep"], rtol=1e-12, atol=1e-12)
            pr = ao.episode_priorities(nets["critic"], nets["target_actor"], nets["target_critic"], e["obs"], e["act"],
                                       e["rew_nstep"], e["term"], burn_in=Bn, learning=L, n_step=n, gamma=gamma)
            assert pr.shape == e["priority"].shape            # E - 60 entries; an episode of exactly 60 steps has none (Q14)
            if pr.size:
                assert rel_l2(pr, e["priority"]) < 2e-5, (ci, rel_l2(pr, e["priority"]))


@pytest.mark.gpu
def test_gpu_actor_priorities_match_reference_fixture():
    from r2d2_b200 import actor_priority as ap
    g = load_golden("ref_actor_prio.npz")
    for ci in range(int(g["n_cases"])):
        (O, A, H, Bn, L, n, gamma), nets, eps = _case(g, ci)
        episodes = [(e["obs"], e["act"], e["rew_raw"], e["term"]) for e in eps]
        prios, rews = ap.episode_priorities(nets["critic"], nets["target_actor"], nets["target_critic"], episodes,
                                            hidden=H, burn_in=Bn, learning=L, n_step=n, gamma=gamma, rewards_are_raw=True)
        for e, pr, rw in zip(eps, prios, rews):
            assert rel_l2(rw, e["rew_nstep"]) < 1e-6                      # n-step sums (episodes of different lengths in one batch)
            assert pr.shape == e["priority"].shape
            if pr.size:
                assert rel_l2(pr, e["priority"]) < 1e-3, (ci, rel_l2(pr, e["priority"]))
