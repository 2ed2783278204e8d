"""numpy restatement (float64 by default) of the learner hot path, written as the SAME
decomposition the CUDA library uses: hoisted input GEMMs -> serial LSTM scan -> head, manual BPTT.

TEST INFRASTRUCTURE: only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may
import this; the product path never does.  Pure numpy, no autograd: every gradient formula that
the CUDA kernels implement is spelled out here and pinned against the real reference's autograd
through tests/golden/*.npz (tests/test_oracle_golden.py).

Reference lines restated
  net forward            models.py:32-40 (actor), :74-83 (critic; tanh at :81 discarded, A outputs)
  LSTMCell gate order    torch.nn.LSTMCell: i, f, g, o; b_ih + b_hh  (used at models.py:37,80)
  burn-in / unroll       learner.py:92-109  (dead actor burn-in learner.py:92 is skipped: its state
                         is dropped at learner.py:117 before any use, quirk Q5)
  n-step target          learner.py:107-108, utils.py:20-21 (h without h^-1, rewards pre-summed)
  critic loss / Adam     learner.py:111-114 (MSE mean over L*B*A; grads flow through burn-in, Q4)
  actor update           learner.py:117-128 (zero state, actor cell stepped twice per row, post-step
                         critic, loss = mean(-Q))
  priorities             learner.py:135-138, utils.py:17-18 (slice [b:-1:B], quirk Q10)
  hard target update     learner.py:63-65,131-132
"""
from __future__ import annotations

import numpy as np

PARAM_KEYS = ("l1.weight", "l1.bias", "l2.weight_ih", "l2.weight_hh", "l2.bias_ih", "l2.bias_hh",
              "l3.weight", "l3.bias")


def _sigmoid(x):
    return 1.0 / (1.0 + np.exp(-x))


def value_rescale(x):
    return np.sign(x) * (np.sqrt(np.abs(x) + 1.0) - 1.0)


def scan_forward(gin, whh, h0, c0, repeat: int = 1):
    """The serial LSTM scan alone.  gin [T,B,4H] = input projection + both biases, whh [4H,H], h0/c0 [B,H].
    steps S = T*repeat; step s consumes row s//repeat.  Returns gates [S,B,4H] post-activation (i,f,g,o) and
    hs, cs [S+1,B,H] (slot 0 = initial state)."""
    T, B, G = gin.shape
    H = G // 4
    S = T * repeat
    hs = np.zeros((S + 1, B, H), gin.dtype)
    cs = np.zeros((S + 1, B, H), gin.dtype)
    gates = np.zeros((S, B, 4 * H), gin.dtype)
    hs[0], cs[0] = h0, c0
    whh_t = whh.T
    for s in range(S):
        g = gin[s // repeat] + hs[s] @ whh_t
        i, f, gg, o = (_sigmoid(g[:, :H]), _sigmoid(g[:, H:2 * H]), np.tanh(g[:, 2 * H:3 * H]),
                       _sigmoid(g[:, 3 * H:]))
        cs[s + 1] = f * cs[s] + i * gg
        hs[s + 1] = o * np.tanh(cs[s + 1])
        gates[s] = np.concatenate((i, f, gg, o), 1)
    return gates, hs, cs


def scan_backward(gates, cs, whh, d_h_head):
    """BPTT of scan_forward.  d_h_head [S,B,H] = dLoss/dh_s from outside the recurrence (zero rows where
    there is none).  Returns d_gates [S,B,4H] (w.r.t. the pre-activations), dh0, dc0 [B,H]."""
    S, B, G = gates.shape
    H = G // 4
    d_gates = np.zeros_like(gates)
    dh_rec = np.zeros((B, H), gates.dtype)
    dc_next = np.zeros((B, H), gates.dtype)
    for s in range(S - 1, -1, -1):
        i, f, gg, o = (gates[s][:, :H], gates[s][:, H:2 * H], gates[s][:, 2 * H:3 * H], gates[s][:, 3 * H:])
        tc = np.tanh(cs[s + 1])
        dh = d_h_head[s] + dh_rec
        d_o = dh * tc * o * (1.0 - o)
        dc = dc_next + dh * o * (1.0 - tc * tc)
        d_i = dc * gg * i * (1.0 - i)
        d_f = dc * cs[s] * f * (1.0 - f)
        d_g = dc * i * (1.0 - gg * gg)
        dc_next = dc * f
        d_gates[s] = np.concatenate((d_i, d_f, d_g, d_o), 1)
        dh_rec = d_gates[s] @ whh
    return d_gates, dh_rec, dc_next


def net_forward(p, x, h0, c0, *, critic: bool, repeat: int = 1):
    """x [T,B,I] -> saved activations.  steps = T*repeat; step s consumes row s//repeat.
    Saved: z1 [T,B,H]; gates [S,B,4H] post-activation (i,f,g,o); hs, cs [S+1,B,H] (slot 0 = initial
    state); out [S,B,A]."""
    z1 = np.tanh(x @ p["l1.weight"].T + p["l1.bias"])
    gin = z1 @ p["l2.weight_ih"].T + (p["l2.bias_ih"] + p["l2.bias_hh"])
    gates, hs, cs = scan_forward(gin, p["l2.weight_hh"], h0, c0, repeat)
    if critic:
        out = hs[1:] @ p["l3.weight"].T + p["l3.bias"]
    else:
        out = np.tanh(np.tanh(hs[1:]) @ p["l3.weight"].T + p["l3.bias"])
    return {"x": x, "z1": z1, "gates": gates, "hs": hs, "cs": cs, "out": out, "repeat": repeat}


def net_backward(p, sv, d_out, *, critic: bool, want_wgrad: bool = True, want_dx: bool = False):
    """Manual BPTT.  d_out [S,B,A] (zero rows where the output is unused)."""
    x, z1, gates, hs, cs, out, repeat = (sv[k] for k in ("x", "z1", "gates", "hs", "cs", "out", "repeat"))
    S, B, _ = d_out.shape
    T = S // repeat
    H = hs.shape[2]
    g = {}
    # weight gradients contract over (step, batch): tensordot runs them as one matrix product each
    wgrad = lambda a, b: np.tensordot(a, b, axes=([0, 1], [0, 1]))  # noqa: E731
    if critic:
        d_pre = d_out
        head_in = hs[1:]
        d_h_head = d_pre @ p["l3.weight"]
    else:
        d_pre = d_out * (1.0 - out * out)
        head_in = np.tanh(hs[1:])
        d_h_head = (d_pre @ p["l3.weight"]) * (1.0 - head_in * head_in)
    if want_wgrad:
        g["l3.weight"] = wgrad(d_pre, head_in)
        g["l3.bias"] = d_pre.sum((0, 1))
    d_gates, dh_rec, dc_next = scan_backward(gates, cs, p["l2.weight_hh"], d_h_head)
    d_gin = d_gates.reshape(T, repeat, B, 4 * H).sum(1)
    if want_wgrad:
        g["l2.weight_hh"] = wgrad(d_gates, hs[:-1])
        g["l2.weight_ih"] = wgrad(d_gin, z1)
        g["l2.bias_ih"] = d_gin.sum((0, 1))
        g["l2.bias_hh"] = g["l2.bias_ih"].copy()
    d_p1 = (d_gin @ p["l2.weight_ih"]) * (1.0 - z1 * z1)
    if want_wgrad:
        g["l1.weight"] = wgrad(d_p1, x)
        g["l1.bias"] = d_p1.sum((0, 1))
    dx = d_p1 @ p["l1.weight"] if want_dx else None
    return g, dx, {"d_gates": d_gates, "d_h_head": d_h_head, "d_p1": d_p1, "dh0": dh_rec, "dc0": dc_next}


def adam_step(p, g, state, lr, b1=0.9, b2=0.999, eps=1e-8):
    """torch.optim.Adam defaults (learner.py:50,52): no weight decay, no amsgrad."""
    state["t"] = state.get("t", 0) + 1
    t = state["t"]
    for k in PARAM_KEYS:
        m = state.setdefault("m/" + k, np.zeros_like(p[k]))
        v = state.setdefault("v/" + k, np.zeros_like(p[k]))
        m *= b1
        m += (1 - b1) * g[k]
        v *= b2
        v += (1 - b2) * g[k] * g[k]
        denom = np.sqrt(v) / np.sqrt(1 - b2 ** t) + eps
        p[k] = p[k] - (lr / (1 - b1 ** t)) * (m / denom)


def td_targets_and_priorities(q, q_next, rew, term, *, burn_in, learning, n_step, gamma, eta=0.9):
    """q, q_next [L,B,A]; rew, term [T',B].  Returns target y [L,B,A], loss, dq, td_sq [L,B], priority [B]."""
    L, B, A = q.shape
    disc = gamma ** n_step
    r = rew[burn_in:burn_in + learning][:, :, None]
    d = term[burn_in + n_step - 1:burn_in + n_step - 1 + learning][:, :, None]
    y = value_rescale(r + disc * (1.0 - d) * q_next)
    diff = q - y
    loss = float(np.mean(diff * diff))
    dq = 2.0 * diff / diff.size
    td_sq = np.mean(diff * diff, axis=2)                      # [L,B]
    flat = td_sq.reshape(-1)                                  # index i*B + b (time-major blocks of B)
    prio = np.zeros(B, q.dtype)
    for b in range(B):
        series = flat[b:-1:B]                                 # learner.py:137; drops the very last element
        prio[b] = eta * series.max() + (1.0 - eta) * series.mean()
    return y, loss, dq, td_sq, prio


class OracleLearner:
    """State (params, Adam moments, step counter) + one iteration of the necessary work."""

    def __init__(self, actor, critic, target_actor=None, target_critic=None, *, burn_in=20, learning=40,
                 n_step=5, gamma=0.997, actor_lr=1e-4, critic_lr=1e-3, target_interval=500,
                 dtype=np.float64):
        cv = lambda d: {k: np.asarray(d[k], dtype=dtype).copy() for k in PARAM_KEYS}  # noqa: E731
        self.actor, self.critic = cv(actor), cv(critic)
        self.target_actor = cv(target_actor if target_actor is not None else actor)
        self.target_critic = cv(target_critic if target_critic is not None else critic)
        self.burn_in, self.learning, self.n_step, self.gamma = burn_in, learning, n_step, gamma
        self.actor_lr, self.critic_lr, self.target_interval = actor_lr, critic_lr, target_interval
        self.dtype = dtype
        self.actor_adam, self.critic_adam = {}, {}
        self.step_count = 0

    def iteration(self, batch, keep=True, grad_hook=None):
        """grad_hook(net_name, grads_dict) may replace gradients in place before the optimiser step (used to
        model the data-parallel all-reduce: mean of per-rank gradients == gradient of the global batch)."""
        dt = self.dtype
        Bn, L, n = self.burn_in, self.learning, self.n_step
        obs, act = np.asarray(batch["obs"], dt), np.asarray(batch["act"], dt)
        T_all, B, _ = obs.shape
        rew = np.asarray(batch["rew"], dt).reshape(T_all, B)
        term = np.asarray(batch["term"], dt).reshape(T_all, B)
        st = {k: np.asarray(batch[k], dt) for k in ("ta_state", "c_state", "tc_state")}
        self.step_count += 1
        # --- target actor over rows [0, Bn+n+L) (learner.py:94,106)
        ta = net_forward(self.target_actor, obs[:Bn + n + L], st["ta_state"][0], st["ta_state"][1], critic=False)
        act_next = ta["out"][Bn + n:]
        # --- target critic: stored actions for burn-in rows, target-actor actions after (learner.py:95,106)
        tc_in = np.concatenate((obs[:Bn + n + L], np.concatenate((act[:Bn + n], act_next), 0)), 2)
        tc = net_forward(self.target_critic, tc_in, st["tc_state"][0], st["tc_state"][1], critic=True)
        q_next = tc["out"][Bn + n:]
        # --- online critic over rows [0, Bn+L) with stored actions (learner.py:93,105)
        c1 = net_forward(self.critic, np.concatenate((obs[:Bn + L], act[:Bn + L]), 2),
                         st["c_state"][0], st["c_state"][1], critic=True)
        q = c1["out"][Bn:]
        y, critic_loss, dq, td_sq, prio = td_targets_and_priorities(
            q, q_next, rew, term, burn_in=Bn, learning=L, n_step=n, gamma=self.gamma)
        d_out = np.concatenate((np.zeros((Bn,) + dq.shape[1:], dt), dq), 0)
        critic_grad, _, _ = net_backward(self.critic, c1, d_out, critic=True)
        if grad_hook is not None:
            grad_hook("critic", critic_grad)
        adam_step(self.critic, critic_grad, self.critic_adam, self.critic_lr)
        # --- actor update (learner.py:117-128)
        zeros = np.zeros((B, self.actor["l2.weight_hh"].shape[1]), dt)
        a1 = net_forward(self.actor, obs[Bn:Bn + L], zeros, zeros, critic=False, repeat=2)
        mu = a1["out"][1::2]                                          # output of the second call per row
        c2 = net_forward(self.critic, np.concatenate((obs[Bn:Bn + L], mu), 2), zeros, zeros, critic=True)
        q_pi = c2["out"]
        actor_loss = float(np.mean(-q_pi))
        dq_pi = np.full(q_pi.shape, -1.0 / q_pi.size, dt)
        _, dx, _ = net_backward(self.critic, c2, dq_pi, critic=True, want_wgrad=False, want_dx=True)
        d_mu = dx[:, :, obs.shape[2]:]
        d_out_a = np.zeros_like(a1["out"])
        d_out_a[1::2] = d_mu
        actor_grad, _, _ = net_backward(self.actor, a1, d_out_a, critic=False)
        if grad_hook is not None:
            grad_hook("actor", actor_grad)
        adam_step(self.actor, actor_grad, self.actor_adam, self.actor_lr)
        if self.step_count % self.target_interval == 0:
            self.target_actor = {k: v.copy() for k, v in self.actor.items()}
            self.target_critic = {k: v.copy() for k, v in self.critic.items()}
        out = {"critic_loss": critic_loss, "actor_loss": actor_loss, "priority": prio,
               "average_td_loss": td_sq.reshape(-1)}
        if keep:
            A = q.shape[2]
            out.update(q_value=q.reshape(-1, A), target_q_value=y.reshape(-1, A), critic_grad=critic_grad,
                       actor_grad=actor_grad, critic_after={k: v.copy() for k, v in self.critic.items()},
                       actor_after={k: v.copy() for k, v in self.actor.items()}, mu=mu, q_pi=q_pi,
                       act_next=act_next, q_next=q_next, d_mu=d_mu)
        return out
