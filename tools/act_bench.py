"""Batched acting on one GPU: r2d2_act_step against the reference's own GPU acting (the four models.py nets called
eagerly through torch at the same batch), and VecActor env-steps/s next to one drop-in CPU Actor.

    python tools/act_bench.py [--steps 2000] [--warmup 200] [--vec-steps 300] [--out DIR]

Prints one JSON line per case, each with the card name and power limit read at start-up.
  kind=lib     median CUDA-event time of one r2d2_act_step (4 launches) per (H, O, A, B); the weight images of the
               four nets (4 * H^2 * 32 bytes) stay L2-resident across steps (126 MB L2; 32 MB at H = 512), so the
               implied weight-image rate is an L2 rate, not an HBM one
  kind=eager   the same step as four torch calls of models.py ActorNet / CriticNet on the same GPU (torch.no_grad)
  kind=vec     VecActor env-steps/s (one vector step = n_envs env steps, host env stepping included) with the
               synthetic env at cfg-3 shape (O=376, A=17, H=512)
  kind=cpu     one drop-in CPU Actor process at the same shape (R2D2_ACTOR_DEVICE=cpu, torch threads as set up)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
from ctypes import c_int, c_void_p

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "pytorch-r2d2-dpg_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

LIB_CASES = ((128, 3, 1), (256, 17, 6), (512, 376, 17))     # BASELINE.json cfg-1/2/3 (H, obs, act)
BATCHES = (1, 8, 64, 256, 1024)


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True, check=True).stdout.strip().split(", ")
    return {"gpu": out[0], "power_limit": out[1] if len(out) > 1 else None}


def nets(O, A, H, device):
    from models import ActorNet, CriticNet
    torch.manual_seed(0)
    d = {"actor": ActorNet(O, A, 0, hidden=H), "target_actor": ActorNet(O, A, 0, hidden=H),
         "critic": CriticNet(O, A, 0, hidden=H), "target_critic": CriticNet(O, A, 0, hidden=H)}
    return {k: v.to(device).eval() for k, v in d.items()}


def time_events(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for a, b in ev:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    t = np.asarray([a.elapsed_time(b) for a, b in ev]) * 1e3
    return float(np.median(t)), float(np.percentile(t, 10)), float(np.percentile(t, 90))


def lib_case(H, O, A, B, steps, warmup, info):
    from r2d2_b200 import native as nv
    from r2d2_b200.actor_priority import _flat
    lib = nv.lib()
    dev = torch.device("cuda:0")
    m = nets(O, A, H, dev)
    h = c_void_p()
    nv.check(lib.r2d2_act_create(nv.byref(h), nv.byref(nv.NetShape(O, A, H, 0)), B))
    try:
        flat = [_flat(m[k].state_dict(), dev) for k in ("actor", "target_actor", "critic", "target_critic")]
        st = nv.current_stream()
        nv.check(lib.r2d2_act_load(h, *(nv.dptr(f) for f in flat), st))
        x = torch.randn(B, O, device=dev)
        s = [torch.zeros(4, 2, B, H, device=dev) for _ in range(2)]
        mu = torch.empty(B, A, device=dev)
        k = [0]

        def step():
            nv.check(lib.r2d2_act_step(h, nv.dptr(x), nv.dptr(s[k[0]]), nv.dptr(s[1 - k[0]]), nv.dptr(mu), B, st))
            k[0] ^= 1
        med, p10, p90 = time_events(step, steps, warmup)
        stt = c_int(0)
        nv.check(lib.r2d2_act_status(h, nv.byref(stt), st))
        w_bytes = 4 * H * H * 32
        rec = dict(info, kind="lib", H=H, obs=O, act=A, B=B, steps=steps, step_us_median=round(med, 2),
                   step_us_p10=round(p10, 2), step_us_p90=round(p90, 2), env_steps_per_s=round(B / med * 1e6, 1),
                   weight_image_bytes_per_step=w_bytes, weight_image_gb_per_s=round(w_bytes / med * 1e-3, 1),
                   weights="L2-resident (4 x H^2 x 32 B images re-read every step)", status=int(stt.value))
    finally:
        lib.r2d2_act_destroy(h)
    print(json.dumps(rec), flush=True)
    return rec


@torch.no_grad()
def eager_case(H, O, A, B, steps, warmup, info):
    dev = torch.device("cuda:0")
    m = nets(O, A, H, dev)
    x = torch.randn(B, O, device=dev)
    for v in m.values():
        v.reset_state()

    def step():                                                  # actor.py:141-144
        a = m["actor"](x)
        ta = m["target_actor"](x)
        m["critic"](x, a)
        m["target_critic"](x, ta)
    med, p10, p90 = time_events(step, steps, warmup)
    rec = dict(info, kind="eager", H=H, obs=O, act=A, B=B, steps=steps, step_us_median=round(med, 2),
               step_us_p10=round(p10, 2), step_us_p90=round(p90, 2), env_steps_per_s=round(B / med * 1e6, 1))
    print(json.dumps(rec), flush=True)
    return rec


def actor_case(kind, n_envs, vec_steps, info):
    os.environ.update(R2D2_OBS_SIZE="376", R2D2_N_ACTIONS="17", R2D2_HIDDEN="512")
    if kind == "cpu":
        os.environ["R2D2_ACTOR_DEVICE"] = "cpu"
    else:
        os.environ.pop("R2D2_ACTOR_DEVICE", None)
    for mname in ("actor", "replay_memory", "models", "utils"):
        sys.modules.pop(mname, None)
    import actor as dropin
    cwd = os.getcwd()
    os.chdir(tempfile.mkdtemp(prefix="act_bench_"))
    os.makedirs("memory_data")
    try:
        a = dropin.Actor(0) if kind == "cpu" else dropin.VecActor(0, n_envs)
        envs = [a.env] if kind == "cpu" else a.envs
        for e in envs:
            e.episode_len = 10 ** 6                              # time the stepping, not episode ends
        steps = vec_steps if kind == "vec" else max(20, vec_steps // 10)
        # warm-up episode of a few steps, then a timed window of `steps` steps
        counter = {"n": 0}
        orig = envs[0].step

        def counted(action):
            counter["n"] += 1
            if counter["n"] >= 4 * (steps + 10):
                raise StopIteration
            if counter["n"] == 4 * 10:
                counter["t0"] = time.perf_counter()
            return orig(action)
        envs[0].step = counted
        try:
            a.run(max_episodes=1)
        except StopIteration:
            pass
        dt = time.perf_counter() - counter["t0"]
        n = 1 if kind == "cpu" else n_envs
        rec = dict(info, kind=kind, H=512, obs=376, act=17, n_envs=n, vector_steps=steps,
                   env_steps_per_s=round(steps * n / dt, 1), torch_threads=torch.get_num_threads())
    finally:
        os.chdir(cwd)
    print(json.dumps(rec), flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--eager-steps", type=int, default=500)
    ap.add_argument("--vec-steps", type=int, default=300)
    ap.add_argument("--out", default=None, help="also write the JSON lines to DIR/act_bench.jsonl")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("act_bench.py measures on a GPU; there is none")
    torch.cuda.set_device(0)
    info = card()
    recs = []
    for H, O, A in LIB_CASES:
        for B in BATCHES:
            recs.append(lib_case(H, O, A, B, args.steps, args.warmup, info))
            recs.append(eager_case(H, O, A, B, args.eager_steps, min(args.warmup, 50), info))
    for n in (1, 16, 64):
        recs.append(actor_case("vec", n, args.vec_steps, info))
    recs.append(actor_case("cpu", 1, args.vec_steps, info))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "act_bench.jsonl"), "w") as f:
            for r in recs:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
