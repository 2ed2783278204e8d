"""Batched GPU acting: one step of the four nets over B environments per call (r2d2_act_* in include/r2d2_b200.h).

The reference steps one environment and runs actor(x), critic(x, mu), target_actor(x), target_critic(x, mu_t) at
batch 1, recording the four (h, c) states from BEFORE the step (/root/reference/actor.py:136-148, 166-167).
ActEngine does the same for B environments in four kernel launches; the states live on the device in the
[4,2,B,H] layout that r2d2_replay_sample gathers (actor, target_actor, critic, target_critic) x (h, c), so the
pre-step state an episode records is exactly the kernel's input.  Noise and clipping stay with the caller.

There is no CPU fallback: without CUDA the constructor raises NativeError.
"""
from __future__ import annotations

from ctypes import c_int, c_void_p

import numpy as np
import torch

from . import native as nv
from .actor_priority import _flat

NET_ORDER = ("actor", "target_actor", "critic", "target_critic")


class ActEngine:
    """B <= max_batch environments in lockstep.  `load(model_dict)` takes the model.pt dict of four state_dicts
    (the format Actor.load_model reads), `reset(mask)` zeroes the state rows of environments that start an episode,
    `step(obs)` returns (mu [B,A], pre-step states [4,2,B,H]) as host arrays."""

    def __init__(self, obs: int, act: int, hidden: int, max_batch: int, device=None):
        if not torch.cuda.is_available():
            raise nv.NativeError("ActEngine needs a CUDA device; there is no CPU fallback")
        self.obs, self.act, self.hidden, self.max_batch = int(obs), int(act), int(hidden), int(max_batch)
        self.device = torch.device(device if device is not None else "cuda:0")
        if self.device.type != "cuda":
            raise nv.NativeError(f"ActEngine runs on a CUDA device, got {self.device}")
        self._lib = nv.lib()
        self._h = c_void_p()
        with torch.cuda.device(self.device):
            nv.check(self._lib.r2d2_act_create(nv.byref(self._h), nv.byref(nv.NetShape(self.obs, self.act, self.hidden, 0)),
                                               self.max_batch))
            # two ping-pong slots [states (8 B H) | mu (B A)]: the pre-step states and this step's mu are one D2H copy
            slot = 8 * self.max_batch * self.hidden + self.max_batch * self.act
            self._slots = [torch.zeros(slot, device=self.device) for _ in range(2)]
            self._obs_d = torch.empty(self.max_batch * self.obs, device=self.device)
        self._obs_h = torch.empty(self.max_batch * self.obs, pin_memory=True)
        self._out_h = torch.empty(slot, pin_memory=True)
        self._cur = 0
        self.batch = self.max_batch
        self._params = None
        self.loaded = False

    # ---- helpers ----
    def _state(self, k: int, B: int | None = None) -> torch.Tensor:
        B = self.batch if B is None else B
        return self._slots[k][:8 * B * self.hidden].view(4, 2, B, self.hidden)

    def _stream(self):
        return c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _set_batch(self, B: int):
        """Re-lay the current state for a different number of environments (rows kept, new rows zero)."""
        if B == self.batch:
            return
        if not 1 <= B <= self.max_batch:
            raise nv.NativeError(f"batch {B} outside [1, {self.max_batch}]")
        old = self._state(self._cur).clone()
        n = min(B, self.batch)
        self._slots[self._cur].zero_()
        self._state(self._cur, B)[:, :, :n] = old[:, :, :n]
        self.batch = B

    # ---- public surface ----
    def load(self, model_dict):
        """model_dict: {'actor', 'target_actor', 'critic', 'target_critic'} -> state_dicts (or dicts of arrays)."""
        with torch.cuda.device(self.device):
            params = [_flat(model_dict[name], self.device) for name in NET_ORDER]
            nv.check(self._lib.r2d2_act_load(self._h, *(nv.dptr(p) for p in params), self._stream()))
        self._params = params             # kept alive until the stream has packed them
        self.loaded = True

    def reset(self, mask=None):
        """Zero the recurrent state of the environments where mask is true (all of them for None): the reference's
        reset_state() at episode start and its lazy zero state (models.py:34-36)."""
        st = self._state(self._cur)
        with torch.cuda.device(self.device):
            if mask is None:
                st.zero_()
            else:
                m = torch.as_tensor(np.asarray(mask, bool).reshape(-1))
                if m.numel() != self.batch:
                    raise nv.NativeError(f"reset mask has {m.numel()} entries, the engine steps {self.batch}")
                idx = torch.nonzero(m).reshape(-1).to(self.device)
                if idx.numel():
                    st.index_fill_(2, idx, 0.0)

    def step(self, obs):
        """obs [B,O] host array -> (mu [B,A] un-noised actor output, states [4,2,B,H] from before this step)."""
        if not self.loaded:
            raise nv.NativeError("ActEngine.step before load()")
        x = np.ascontiguousarray(obs, dtype=np.float32)
        if x.ndim != 2 or x.shape[1] != self.obs:
            raise nv.NativeError(f"obs must be [B,{self.obs}], got {x.shape}")
        B = x.shape[0]
        self._set_batch(B)
        H, A = self.hidden, self.act
        n_st = 8 * B * H
        cur, nxt = self._slots[self._cur], self._slots[1 - self._cur]
        self._obs_h[:B * self.obs].numpy()[:] = x.reshape(-1)
        with torch.cuda.device(self.device):
            self._obs_d[:B * self.obs].copy_(self._obs_h[:B * self.obs], non_blocking=True)
            nv.check(self._lib.r2d2_act_step(self._h, nv.dptr(self._obs_d), nv.dptr(cur), nv.dptr(nxt),
                                             c_void_p(cur.data_ptr() + 4 * n_st), B, self._stream()))
            self._out_h[:n_st + B * A].copy_(cur[:n_st + B * A], non_blocking=True)
            torch.cuda.current_stream(self.device).synchronize()
        self._cur = 1 - self._cur
        out = self._out_h[:n_st + B * A].numpy()
        return out[n_st:].reshape(B, A).copy(), out[:n_st].reshape(4, 2, B, H).copy()

    def state(self) -> np.ndarray:
        """The current (post-step) state [4,2,B,H] as a host array."""
        return self._state(self._cur).cpu().numpy()

    def status(self) -> int:
        st = c_int(0)
        with torch.cuda.device(self.device):
            nv.check(self._lib.r2d2_act_status(self._h, nv.byref(st), self._stream()))
        return int(st.value)

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            try:
                torch.cuda.synchronize(self.device)
            except Exception:
                pass
            self._lib.r2d2_act_destroy(self._h)
            self._h = c_void_p()

    def __del__(self):
        self.close()
