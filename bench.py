#!/usr/bin/env python
"""bench.py - learner sequence-steps/sec (batch x seq_len per learner iteration) of the B200-native learner hot
path.  Headline workload = BASELINE.json configs[2], the largest single-GPU configuration: synthetic Humanoid
shape obs=376 act=17 hidden=512 seq_len=80 burn_in=40 batch=512 PER GPU (weak scaling: every rank owns a replay
shard in HBM and a batch of 512; the two flat gradient blocks are all-reduced over NCCL at the optimiser steps).

  python bench.py --gpus N --steps K --warmup W          # torchrun launches one process per GPU for N > 1
  python bench.py --impl reference ...                   # the reference's CPU implementation (oracle port)
  python bench.py --config cfg2|cfg1                     # BASELINE.json configs[1] / configs[0] shapes
  python bench.py --config replay                        # configs[3]: 250k stored sequence starts per GPU, sample / update
  python bench.py --dump-outputs DIR                     # also write the last timed step's outputs (Arm.dump_outputs)

A step = one pass of learner.py:84-139: prioritized sample from the HBM replay shard -> gather -> target/online
chains -> TD/priority kernels -> critic BPTT + Adam -> actor chain -> DPG backward + Adam -> priority write-back into
the sum tree.  One JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "pytorch-r2d2-dpg_b200")
for _p in (ROOT, PKG):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

CONFIGS = {
    # BASELINE.json configs[0] shapes (reference as-is, walker sizes) / configs[1] / configs[2] (headline)
    "cfg1": dict(obs=24, act=6, hidden=128, batch=32, burn_in=20, learning=40, n_step=5),
    "cfg2": dict(obs=17, act=6, hidden=256, batch=256, burn_in=40, learning=80, n_step=5),
    "cfg3": dict(obs=376, act=17, hidden=512, batch=512, burn_in=40, learning=80, n_step=5),
}
METRIC = "learner sequence-steps/sec (batch x seq_len)"
DTYPE = "bf16x3 (fp32 operands split into bf16 hi+lo, three tensor-core passes, fp32 accumulate: ~16-bit operands)"


def workload_string(name, c):
    """identical in both arms (the driver compares them)"""
    return f"{name}: " + " ".join(f"{k}={v}" for k, v in c.items())


def lstm_flops_per_iteration(c):
    """SURVEY 8d: FLOP_lstm = 16*B*H^2*(5*Bn + 13*L + 2*n) (necessary cell-steps, fwd + bwd)."""
    return 16.0 * c["batch"] * c["hidden"] ** 2 * (5 * c["burn_in"] + 13 * c["learning"] + 2 * c["n_step"])


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        d = json.load(open(path))
        return {"bf16_burst": d["bf16_tflops"], "bf16_sustained": d["bf16_tflops_sustained"], "hbm": d["hbm_gbs"],
                "source": "measured"}
    return {"bf16_burst": 1590.0, "bf16_sustained": 1400.0, "hbm": 6650.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi sampling DURING the timed region (B200_PROFILING.md clocks line)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc, self.t0, self.t1 = index, [], None, None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "50"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def mark(self, begin):
        """wall-clock window of the timed region: only samples taken inside it are reported"""
        if begin:
            self.t0 = time.time()
        else:
            self.t1 = time.time()

    def stop(self):
        if self.proc is not None:
            time.sleep(0.06)
            self.proc.terminate()
        inside = [r for t, r in self.rows if self.t0 is not None and self.t0 <= t <= (self.t1 or 1e30) + 0.05]
        rows = inside if inside else [r for _, r in self.rows[-3:]]
        sm = [float(r[0]) for r in rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i] == "Active" for r in rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def build_replay(engine, cfg, n_episodes, episode_len, seed, device):
    """Per-GPU replay shard with synthetic episodes.  One episode's arrays are generated per 16 episodes (fresh
    priorities every time): the content of a row does not change what a step costs."""
    rng = np.random.default_rng(seed)
    n_rows = episode_len + cfg.n_step
    rp = engine.DeviceReplay(cfg, capacity_rows=n_episodes * n_rows, device=device)
    for e in range(n_episodes):
        if e % 16 == 0:
            term = np.zeros(n_rows, np.float32)
            term[episode_len:] = 1
            obs = rng.standard_normal((n_rows, cfg.obs), dtype=np.float32)
            act = rng.uniform(-1, 1, (n_rows, cfg.act)).astype(np.float32)
            rew = rng.standard_normal(n_rows, dtype=np.float32)
            obs[episode_len:] = 0
            act[episode_len:] = 0
            rew[episode_len:] = 0
            states = 0.1 * rng.standard_normal((episode_len, 4, 2, cfg.hidden), dtype=np.float32)
        prio = rng.uniform(0.01, 1.0, episode_len - (cfg.burn_in + cfg.learning)).astype(np.float32)
        rp.add_episode(obs, act, rew, term, states, prio)
    return rp


def log(msg):
    print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


def cpu_model():
    """CPU model string of the host the CPU baseline ran on (SURVEY 8d asks for it next to os.cpu_count())."""
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.lower().startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def pick_cpu_threads(name, c):
    """Thread count of the CPU arms.  torch CPU ops of this size stop scaling - and can collapse - long before a
    100+ core box is full, so FULL-BATCH port iterations (all phases: sample, chains, BPTT, Adam; a shortened window
    so that a probe iteration costs ~1/10 of a real one) are timed for a few candidates and the fastest is kept.  The
    choice is cached per (CPU model, core count, config) in /tmp so that `--impl reference` and the `cpu_baseline` leg
    of the B200 arm, which run back to back on one box, use the same setting (round 1: a 12-step LSTMCell probe flipped
    between 16 and 32 threads from run to run and moved the reference arm by 2.8x)."""
    ncpu = os.cpu_count() or 1
    key = f"{cpu_model()}|{ncpu}|{name}"
    cache_path = "/tmp/r2d2_b200_cpu_threads.json"
    try:
        cache = json.load(open(cache_path))
    except Exception:
        cache = {}
    if key in cache:
        log(f"cpu threads: {cache[key]['threads']} (cached choice of this box: {cache[key]['probe']})")
        return int(cache[key]["threads"])
    from oracle import ref_port
    cands = sorted({t for t in (8, 16, 32, 64) if t <= ncpu}) or [ncpu]
    small = dict(c, burn_in=2, learning=6, n_step=2)
    pc = ref_port.PathConfig(**small)
    probe = {}
    for t in cands:
        torch.set_num_threads(t)
        lr = ref_port.PortLearner(pc, seed=1)
        batch = ref_port.synthetic_batch(pc, seed=0)
        ts = []
        for rep in range(3):
            t0 = time.perf_counter()
            lr.iteration(batch, keep_tensors=False)
            ts.append(time.perf_counter() - t0)
        probe[t] = min(ts[1:])
        log(f"cpu thread probe: {t} threads -> {probe[t] * 1e3:.0f} ms per shortened full-batch iteration")
        if probe[t] > 2.0 * min(probe.values()):
            break  # past the knee: more threads only add contention
    best = min(probe, key=probe.get)
    cache[key] = {"threads": best, "probe": {str(k): round(v, 4) for k, v in probe.items()}}
    try:
        json.dump(cache, open(cache_path, "w"))
    except OSError:
        pass
    return best


def time_cpu_port(name, c, steps, warmup, budget_s):
    """The reference's CPU implementation of the path (oracle/ref_port.py: same torch CPU operators, python loops,
    autograd, Adam, two-level WeightedRandomSampler draw) on this box's host cores, full batch, full window.
    Stops early (after >= 1 timed iteration) when `budget_s` of wall clock is spent."""
    from oracle import ref_port
    threads = pick_cpu_threads(name, c)
    torch.set_num_threads(threads)
    pc = ref_port.PathConfig(**c)
    lr = ref_port.PortLearner(pc, seed=1)
    rp = ref_port.synthetic_replay(pc, n_episodes=max(8, (2 * c["batch"]) // 100 + 8), episode_len=250, seed=0)
    times, t_start = [], time.perf_counter()
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        ep, sq, batch = rp.sample()
        out = lr.iteration(batch, keep_tensors=False)
        rp.write_back(ep, sq, out["priority"])
        if i >= warmup:
            times.append(time.perf_counter() - t0)
        log(f"cpu port iteration {i}: {time.perf_counter() - t0:.2f} s")
        if times and time.perf_counter() - t_start > budget_s:
            break
    sec = float(np.median(times))
    return c["batch"] * c["learning"] / sec, sec, threads, len(times)


def run_reference(args, name, c):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    warm = 1   # a CPU iteration takes seconds: one untimed iteration warms allocator and thread pool
    value, sec, threads, done = time_cpu_port(name, c, args.steps, warm, budget_s=200.0)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "seq-steps/s", "n_gpus": args.gpus,
            "steps": args.steps, "steps_timed": done, "warmup": args.warmup, "warmup_run": warm,
            "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_string(name, c),
                       "note": "reference CPU learner (oracle/ref_port.py port; /root/reference is python and not "
                               "present on this box), full batch and full window per step; a step is one learner "
                               "iteration (seconds on the host): at most 200 s of them are timed (steps_timed, median), "
                               "the rate does not depend on the count"},
            "cpu_baseline": {"value": value, "unit": "seq-steps/s", "cores": threads, "kind": "port",
                             "sample": f"{done} full learner iterations at batch {c['batch']} after {warm} warm-up, "
                                       f"{threads} torch threads (fastest of a full-batch probe over {os.cpu_count()} host cores)",
                             "cpu_model": cpu_model(), "host_cores": os.cpu_count()},
            "e2e": {"value": value, "unit": "seq-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


_REAL_STDOUT = None


def _claim_stdout():
    """stdout must carry exactly ONE JSON line: point fd 1 at stderr for everything libraries print (NCCL / c10d
    banners go to fd 1 of every rank) and keep the real stdout for emit()."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


class Arm:
    """engine + replay shard of one configuration, and the two timed loops (HBM-resident and host-fed)."""

    def __init__(self, engine_mod, c, dev, rank, episodes, data_parallel, seed_base=100):
        self.engine_mod, self.c, self.dev = engine_mod, c, dev
        self.cfg = engine_mod.PathConfig(**c)
        self.eng = engine_mod.LearnerEngine(self.cfg, device=dev, seed=1)
        if data_parallel:
            self.eng.enable_data_parallel()
        self.ep_len = 250
        self.episodes = episodes
        self.rp = build_replay(engine_mod, self.cfg, episodes, self.ep_len, seed=seed_base + rank, device=dev)
        self.gen = torch.Generator(device=dev).manual_seed(1234 + rank)
        # what the resident loop writes back into the tree: see _next_batch
        self.written_prio = 0.01 + 0.99 * torch.rand(self.cfg.batch, device=dev,
                                                     generator=torch.Generator(device=dev).manual_seed(4321 + rank))

    def _next_batch(self, eng, used):
        """LearnerEngine.step's prefetch hook: tree write-back of the batch just used (learner.py:136-139), then the
        sum-tree draw + gather of the next one (learner.py:84) - the same work per iteration as the sequential loop,
        issued as soon as the priorities exist so that the next batch's target chains can run mid-iteration.

        The write-back scatters a fixed, seeded priority vector into the trained leaves rather than the priorities the
        step computed: the same kernel, element count and bytes, so the same cost.  Computed priorities carry the
        rounding of the build (split-K and reduction atomics), and written back they would steer every later draw:
        two runs, or two builds, would train on different batches after a few dozen steps.  This way the batches
        depend on the seeds alone and the outputs of any step can be compared (dump_outputs)."""
        self.rp.update_priorities(used.leaf_idx, self.written_prio)
        self.trained_leaf_idx = used.leaf_idx    # slot of the batch just trained on: the next draw fills the other one
        self.rp.sample_into(eng, generator=self.gen)

    def step_resident(self):
        self.eng.step(prefetch=self._next_batch)

    def time_resident(self, steps, warmup, barrier, clocks=None):
        self.eng.discard_prefetched()
        self.rp.sample_into(self.eng, generator=self.gen)     # batch 0; every step draws its successor
        for _ in range(warmup):
            self.step_resident()
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        if clocks is not None:
            clocks.mark(True)
        ev0.record()
        for _ in range(steps):
            self.step_resident()
        ev1.record()
        barrier()
        if clocks is not None:
            clocks.mark(False)
        return ev0.elapsed_time(ev1) / steps

    def time_host_fed(self, steps, warmup, barrier):
        """e2e: the whole iteration - sum-tree draw + gather, learner phases, tree write-back - with the step's batch
        ALSO arriving from pinned HOST memory (the reference's boundary: replay_memory.py:123-133 builds the batch on
        the host and copies it to the device every iteration) and the priorities / losses read back to the host with
        a stream synchronisation (learner.py:135).  The host batch overwrites the device-gathered one, so the timed
        region contains both the device sampler work and the host->device traffic of the same bytes."""
        eng, rp = self.eng, self.rp
        eng.discard_prefetched()
        B = self.cfg.batch
        n_pool = 3
        pool = []
        for _ in range(n_pool):
            rp.sample_into(eng, generator=self.gen)
            torch.cuda.synchronize()
            pool.append({k: getattr(eng, k).cpu().pin_memory() for k in ("obs", "act", "rew", "term", "states")})
        host_prio = torch.empty(B, dtype=torch.float32).pin_memory()
        host_loss = torch.empty(2, dtype=torch.float32).pin_memory()
        h2d = sum(v.numel() * 4 for v in pool[0].values())
        d2h = (B + 2) * 4
        keys = list(pool[0].keys())
        copy_stream = torch.cuda.Stream()
        stage = [{k: torch.empty_like(getattr(eng, k)) for k in keys} for _ in range(2)]
        ready = [torch.cuda.Event() for _ in range(2)]
        consumed = [torch.cuda.Event() for _ in range(2)]
        for e in consumed:
            e.record(torch.cuda.current_stream())

        def prefetch(i):     # pinned batch of step i crosses PCIe on a copy stream while step i-1 computes
            s_ = i % 2
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(consumed[s_])
                for k, v in pool[i % n_pool].items():
                    stage[s_][k].copy_(v, non_blocking=True)
                ready[s_].record(copy_stream)

        def fill(i):         # batch i: device sampler, then the host-built batch of the same shape over it
            s_ = i % 2
            cur = torch.cuda.current_stream()
            rp.sample_into(eng, generator=self.gen)               # sum-tree draw + gather (device sampler, learner.py:84)
            cur.wait_event(ready[s_])
            for k in keys:                                        # H2D ran on the copy stream; this is the on-device hand-over
                getattr(eng, k).copy_(stage[s_][k], non_blocking=True)
            consumed[s_].record(cur)
            prefetch(i + 1)

        def step_host(i):
            cur = torch.cuda.current_stream()

            def next_batch(eng_, used):
                rp.update_priorities(used.leaf_idx, used.priority)    # learner.py:136-139
                fill(i + 1)

            eng.step(prefetch=next_batch)
            host_prio.copy_(eng.priority, non_blocking=True)
            host_loss.copy_(eng.losses, non_blocking=True)
            cur.synchronize()                                     # the host consumes the priorities every iteration

        prefetch(0)
        fill(0)
        for i in range(warmup):
            step_host(i)
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for i in range(warmup, warmup + steps):
            step_host(i)
        ev1.record()
        barrier()
        copy_stream.synchronize()
        return ev0.elapsed_time(ev1) / steps, h2d, d2h

    def dump_outputs(self, out_dir):
        """What the last resident step handed its caller, as DIR/<name>.npy: q / target / squared TD / priorities /
        losses of the iteration, the actor and critic weights after its updates, and the replay rows it trained on
        (float64 indices).  About 25 MB at cfg3, the largest configuration.

        Replay shard, weights, uniforms and the priorities written back are seeded (_next_batch), so runs with the
        same arguments train on the same batches; their outputs differ by the rounding of the atomics only."""
        self.eng.flush()
        torch.cuda.synchronize()
        eng = self.eng
        arrays = {"q_value": eng.q_value, "target_q_value": eng.target_q_value, "td_sq": eng.td_sq,
                  "priority": eng.priority, "losses": eng.losses, "actor_params": eng.flat["actor"],
                  "critic_params": eng.flat["critic"], "leaf_idx": self.trained_leaf_idx.double()}
        os.makedirs(out_dir, exist_ok=True)
        for name, t in arrays.items():
            np.save(os.path.join(out_dir, name + ".npy"), t.detach().cpu().numpy())

    @property
    def launches_per_step(self):
        return self.eng.launches_per_iteration + 2 + 1   # + tree_sample, gather_batch + tree_update

    def close(self):
        self.rp.close()
        self.eng.close()


def scan_roofline(nv, c, dev, peaks, ms_iter):
    """Roofline of the dominant kernel: the persistent LSTM scan (the serial h*W_hh^T half of every cell step;
    the hoisted x*W_ih^T half runs in gemm_f32).  Algorithmic FLOPs per launch = 2*B*H*4H per cell step x S steps.
    Forward and BPTT kernels are timed alone with CUDA events on the launch stream."""
    B, H = c["batch"], c["hidden"]
    S = c["burn_in"] + c["n_step"] + c["learning"]
    gin = torch.randn(S, B, 4 * H, device=dev) * 0.5
    whh = (torch.rand(4 * H, H, device=dev) * 2 - 1) / np.sqrt(4 * H)
    gates = torch.empty_like(gin)
    hs = torch.empty(S + 1, B, H, device=dev)
    cs = torch.empty(S + 1, B, H, device=dev)
    dh = torch.randn(S, B, H, device=dev) * 0.01
    lib, st = nv.lib(), nv.current_stream()
    scratch = torch.empty(B * 4 * H + 64, device=dev)

    def fwd():
        nv.check(lib.r2d2_lstm_scan_forward(nv.dptr(gin), nv.dptr(whh), None, None, nv.dptr(gates), nv.dptr(hs),
                                            nv.dptr(cs), None, S, B, H, 1, nv.dptr(scratch), st))

    def bwd():
        nv.check(lib.r2d2_lstm_scan_backward(nv.dptr(gates), nv.dptr(hs), nv.dptr(cs), nv.dptr(whh), nv.dptr(dh), 0,
                                             nv.dptr(gates), nv.dptr(gates), S, B, H, 1, nv.dptr(scratch), st))
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    out = {}
    for name, fn in (("fwd", fwd), ("bwd", bwd)):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        reps = 5
        ev0.record()
        for _ in range(reps):
            fn()
        ev1.record()
        torch.cuda.synchronize()
        out[name] = ev0.elapsed_time(ev1) / reps
    scan_flops = 2.0 * B * H * 4 * H * S
    achieved = scan_flops / (out["fwd"] * 1e-3) / 1e12
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "r02_scan_fwd_traffic.json")
    if os.path.isfile(tpath):
        try:
            traffic = json.load(open(tpath)).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    kname = ("lstm_scan_fwd_big_kernel (H=512: cluster of 16, 7 resident clusters x <=80 rows as two ping-pong sub-tiles, "
             "W_hh in TMEM + smem tail, h_t all-gather through L2 multicast)") if H == 512 else \
        "lstm_scan_fwd_pp_kernel (persistent cluster LSTM scan, tcgen05 ping-pong over two row sub-tiles, W_hh in TMEM)"
    flops_it = lstm_flops_per_iteration(c)
    return {"kernel": kname + f", {S} cell steps", "bound": "tensor", "achieved": achieved, "peak": peaks["bf16_burst"],
            "unit": "TFLOP/s", "frac": achieved / peaks["bf16_burst"], "traffic": traffic,
            "traffic_source": "profiles/r02_scan_fwd_traffic.json (ncu --set full of this kernel, dram read + write per launch)"
            if traffic else None,
            "peak_source": peaks["source"] + " bf16 dense burst (kernel timed alone)",
            "us_per_step": out["fwd"] * 1e3 / S,
            "bptt_kernel": {"us_per_step": out["bwd"] * 1e3 / S,
                            "achieved_tflops": scan_flops / (out["bwd"] * 1e-3) / 1e12,
                            "frac": scan_flops / (out["bwd"] * 1e-3) / 1e12 / peaks["bf16_burst"]},
            "whole_iteration": {"lstm_flops": flops_it, "achieved_tflops": flops_it / (ms_iter * 1e-3) / 1e12,
                                "frac_of_sustained_peak": flops_it / (ms_iter * 1e-3) / 1e12 / peaks["bf16_sustained"]}}


def dump_replay_outputs(out_dir, rp, eng, n_cols=64):
    """What the replay legs hand their caller, as DIR/<name>.npy: the last timed draw (leaf indices, float64, and
    the gathered batch of a fixed, seeded sample of n_cols of its sequences - the whole batch is ~100 MB at cfg3) and
    the tree after the timed priority updates (its total, float64, and its level above the leaves)."""
    torch.cuda.synchronize()
    cols = np.sort(np.random.default_rng(0).choice(eng.cfg.batch, n_cols, replace=False))
    idx = torch.as_tensor(cols, device=eng.leaf_idx.device)
    arrays = {"leaf_idx": eng.leaf_idx.double(), "obs": eng.obs[:, idx], "act": eng.act[:, idx], "rew": eng.rew[:, idx],
              "term": eng.term[:, idx], "states": eng.states[:, :, idx], "tree_level1": rp.tree_level(1),
              "total_priority": torch.tensor([rp.stats()["total_priority"]], dtype=torch.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().cpu().numpy())


def run_replay_bench(args, engine, dev, world, rank, dist, barrier):
    """BASELINE.json configs[3]: GPU-resident prioritized replay, 2 M stored sequence starts sharded 8-way = 250 k starts
    per GPU (1000 episodes x 250 starts, Humanoid row widths): sum-tree sample + gather and priority-update throughput,
    index bit-exactness against the C restatement of the tree (oracle/sumtree_oracle.c) - checker only."""
    from oracle.sumtree import SumTreeOracle
    c = CONFIGS["cfg3"]
    cfg = engine.PathConfig(**c)
    n_ep, starts = 1000, 250
    E = starts + cfg.burn_in + cfg.learning
    n_rows = E + cfg.n_step
    rp = engine.DeviceReplay(cfg, capacity_rows=n_ep * n_rows, device=dev)
    oracle = SumTreeOracle(n_ep * n_rows) if rank == 0 else None
    rng = np.random.default_rng(rank)
    t0 = time.time()
    obs = rng.standard_normal((n_rows, cfg.obs), dtype=np.float32)
    act = rng.uniform(-1, 1, (n_rows, cfg.act)).astype(np.float32)
    rew = rng.standard_normal(n_rows, dtype=np.float32)
    term = np.zeros(n_rows, np.float32)
    term[E:] = 1
    st = 0.1 * rng.standard_normal((E, 4, 2, cfg.hidden), dtype=np.float32)
    for e in range(n_ep):
        p = rng.uniform(0.01, 1.0, starts).astype(np.float32)
        rp.add_episode(obs, act, rew, term, st, p)
        if oracle is not None:
            oracle.set_range(e * n_rows, p)
    torch.cuda.synchronize()
    ingest_s = time.time() - t0
    eng = engine.LearnerEngine(cfg, device=dev)
    gen = torch.Generator(device=dev).manual_seed(rank)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    B = cfg.batch
    steps, warm = args.steps, max(args.warmup, 5)
    for _ in range(warm):
        rp.sample_into(eng, generator=gen)
    barrier()
    ev0.record()
    for _ in range(steps):
        rp.sample_into(eng, generator=gen)
    ev1.record()
    barrier()
    ms_sample = ev0.elapsed_time(ev1) / steps
    u = torch.rand(1 << 20, device=dev, generator=gen)
    for _ in range(3):
        leaf = rp.sample_indices(u)
    ev0.record()
    for _ in range(10):
        leaf = rp.sample_indices(u)
    ev1.record()
    torch.cuda.synchronize()
    draws_per_s = 10 * u.numel() / (ev0.elapsed_time(ev1) * 1e-3)
    exact = exact_after = None
    if rank == 0:   # same uniforms, same tree: identical flat indices from the CUDA tree and its C restatement
        exact = bool(np.array_equal(leaf.cpu().numpy(), oracle.sample(u.cpu().numpy())))
    prio = torch.rand(B, device=dev, generator=gen)
    for _ in range(warm):
        rp.update_priorities(eng.leaf_idx, prio)
    barrier()
    ev0.record()
    for _ in range(steps):
        rp.update_priorities(eng.leaf_idx, prio)
    ev1.record()
    barrier()
    ms_update = ev0.elapsed_time(ev1) / steps
    if rank == 0:   # and again after a batch of priority writes (duplicates: last writer wins in both)
        oracle.update_batch(eng.leaf_idx.cpu().numpy(), prio.cpu().numpy())
        u2 = torch.rand(100000, device=dev, generator=gen)
        exact_after = bool(np.array_equal(rp.sample_indices(u2).cpu().numpy(), oracle.sample(u2.cpu().numpy())))
    if args.dump_outputs and rank == 0:
        dump_replay_outputs(args.dump_outputs, rp, eng)
    t = torch.tensor([ms_sample, ms_update], device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_sample, ms_update = float(t[0]), float(t[1])
    batch_bytes = 4 * (cfg.rows * B * (cfg.obs + cfg.act + 2) + 8 * B * cfg.hidden)
    peaks = measured_peaks()
    if rank == 0:
        emit({"metric": "replay sampled sequences/sec (sum-tree draw + time-major gather)", "value": world * B / (ms_sample * 1e-3),
              "unit": "sequences/s", "n_gpus": world, "steps": steps, "warmup": warm, "ms_per_step": ms_sample,
              "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 data, fp32 tree sums, int64 indices",
              "data": "synthetic",
              "config": {"workload": f"replay: {n_ep * starts} stored sequence starts per GPU ({n_ep} episodes x {n_rows} rows, "
                                     f"obs={cfg.obs} act={cfg.act} hidden={cfg.hidden}), batch {B} x {cfg.rows} rows per draw",
                         "total_starts": world * n_ep * starts},
              "updates_per_s": world * B / (ms_update * 1e-3), "update_us_per_batch": ms_update * 1e3,
              "sample_gather_us_per_batch": ms_sample * 1e3, "tree_draws_per_s_rank0": draws_per_s,
              "indices_bit_exact_vs_c_tree": exact, "indices_bit_exact_after_update": exact_after,
              "ingest_s_per_shard": round(ingest_s, 2),
              "roofline": {"kernel": "gather_batch_kernel (+ tree_sample_kernel)", "bound": "hbm",
                           "achieved": 2 * batch_bytes / (ms_sample * 1e-3) / 1e9, "peak": peaks["hbm"], "unit": "GB/s",
                           "frac": 2 * batch_bytes / (ms_sample * 1e-3) / 1e9 / peaks["hbm"], "traffic": None,
                           "algorithmic_bytes": 2 * batch_bytes, "peak_source": peaks["source"] + " copy bandwidth"},
              "gpu_launches": 3 * steps})


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100,
                    help="timed steps of every leg (headline, host-fed, strong-scaling, secondary configs, replay)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="cfg3", choices=sorted(CONFIGS) + ["replay"])
    ap.add_argument("--episodes", type=int, default=384, help="episodes in the per-GPU replay shard")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--no-extras", action="store_true", help="skip the secondary configs / strong-scaling legs (profiling runs)")
    ap.add_argument("--cpu-steps", type=int, default=4)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (rank 0), to compare two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        # the CPU port stops on a wall-clock budget: how many iterations it ran, and so its last outputs, vary
        ap.error("--dump-outputs writes the outputs of the B200 arm: not with --impl reference")
    if args.warmup < 3:
        args.warmup = 3
    name = args.config if args.config != "replay" else "cfg3"
    c = CONFIGS[name]
    if args.impl == "reference":
        return run_reference(args, name, c)

    from r2d2_b200 import engine, native as nv
    from r2d2_b200.dist_env import DistEnv

    env = DistEnv.from_environ()
    world, rank, local = env.world, env.rank, env.local_rank
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    dist = None
    if world > 1:
        # stdout carries exactly one JSON line: keep NCCL's banner / debug output out of it
        os.environ.setdefault("NCCL_DEBUG_FILE", "/tmp/nccl_bench_%h_%p.log")
        dist = env.init_process_group("nccl", device=dev)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    if args.config == "replay":
        run_replay_bench(args, engine, dev, world, rank, dist, barrier)
        if dist is not None:
            dist.destroy_process_group()
        return

    log(f"world={world} rank={rank}: building engine + replay shard ({name})")
    arm = Arm(engine, c, dev, rank, args.episodes, data_parallel=True)
    cfg = arm.cfg
    B, L = cfg.batch, cfg.learning
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()          # started before the warm-up so that samples exist when the timed region begins
    log("HBM-resident arm")
    ms = arm.time_resident(args.steps, args.warmup, barrier, clocks)
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        arm.dump_outputs(args.dump_outputs)

    def max_over_ranks(x):
        t = torch.tensor([x], device=dev)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    ms_per_rank = [ms]
    if dist is not None:   # every rank's own device time of the timed loop (they run in lock step through the all-reduces)
        g = [torch.zeros(1, device=dev) for _ in range(world)]
        dist.all_gather(g, torch.tensor([ms], device=dev))
        ms_per_rank = [round(float(x.item()), 4) for x in g]
    ms = max_over_ranks(ms)
    value = world * B * L / (ms * 1e-3)
    log(f"resident arm: {ms:.3f} ms/step; host-fed (e2e) arm")
    ms_e2e, h2d, d2h = arm.time_host_fed(args.steps, args.warmup, barrier)
    ms_e2e = max_over_ranks(ms_e2e)
    e2e_value = world * B * L / (ms_e2e * 1e-3)
    replicas_identical = arm.eng.replicas_identical() if world > 1 else None
    launches_per_step = arm.launches_per_step

    log("roofline: timing the scan kernels alone")
    peaks = measured_peaks()
    roofline = scan_roofline(nv, c, dev, peaks, ms)

    # ---- strong scaling (SURVEY 8e): the configuration's batch is the GLOBAL batch, B/N sequences per GPU
    strong = None
    if world > 1 and not args.no_extras and B % world == 0:
        log("strong-scaling leg")
        cs = dict(c, batch=B // world)
        arm_s = Arm(engine, cs, dev, rank, max(64, args.episodes // world), data_parallel=True, seed_base=500)
        ms_s = max_over_ranks(arm_s.time_resident(args.steps, args.warmup, barrier))
        strong = {"global_batch": B, "per_gpu_batch": B // world, "ms_per_step": ms_s,
                  "value": B * L / (ms_s * 1e-3), "unit": "seq-steps/s",
                  "replicas_identical": arm_s.eng.replicas_identical()}
        arm_s.close()
    # ---- the other BASELINE configs on the same build (per GPU batch as configured; same timed loop, fewer steps)
    others = {}
    if not args.no_extras:
        for oname in ("cfg2", "cfg1"):
            if oname == name:
                continue
            log(f"secondary config {oname}")
            arm_o = Arm(engine, CONFIGS[oname], dev, rank, 128, data_parallel=True, seed_base=900)
            ms_o = max_over_ranks(arm_o.time_resident(args.steps, args.warmup, barrier))
            co = CONFIGS[oname]
            others[oname] = {"workload": workload_string(oname, co), "ms_per_step": ms_o,
                             "value": world * co["batch"] * co["learning"] / (ms_o * 1e-3), "unit": "seq-steps/s",
                             "gpu_launches_per_step": arm_o.launches_per_step}
            arm_o.close()

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        log("cpu_baseline leg (oracle port on host cores)")
        v, sec, threads, done = time_cpu_port(name, c, args.cpu_steps, 1, budget_s=45.0)
        cpu_baseline = {"value": v, "unit": "seq-steps/s", "cores": threads, "kind": "port",
                        "sample": f"{done} full learner iterations at batch {B} after 1 warm-up ({sec:.2f} s each, median), "
                                  f"{threads} torch threads (fastest of a full-batch probe over {os.cpu_count()} host cores; "
                                  f"same choice as --impl reference on this box)",
                        "cpu_model": cpu_model(), "host_cores": os.cpu_count()}
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "seq-steps/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": DTYPE, "data": "synthetic",
                "config": {"workload": workload_string(name, c), "per_gpu": True,
                           "parallelism": f"dp{world}", "global_batch": world * B,
                           "replay_shard": f"{args.episodes} episodes x {arm.ep_len + cfg.n_step} rows per GPU in HBM",
                           "l2": "inputs larger than L2: every step streams several GB of activations and gathers its batch "
                                 "from a multi-GB replay shard"},
                "e2e": {"value": e2e_value, "unit": "seq-steps/s", "ms_per_step": ms_e2e, "h2d_bytes_per_step": h2d,
                        "d2h_bytes_per_step": d2h,
                        "feed": "per step: sum-tree draw + gather on the device, the step's batch copied from PINNED HOST memory "
                                "(copy stream, overlaps the previous step) over the gathered one, learner iteration, tree "
                                "write-back, priorities + losses read back to the host and the stream synchronised "
                                "(write-back of batch i and draw + host copy of batch i+1 are issued as soon as the "
                                "priorities of batch i exist: LearnerEngine.step(prefetch=...))"},
                "iterations_per_s": world * 1e3 / ms, "rows_per_s": world * B * (cfg.burn_in + L) / (ms * 1e-3),
                "gpu_launches": launches_per_step * args.steps, "gpu_launches_per_step": launches_per_step,
                "roofline": roofline, "cpu_baseline": cpu_baseline, "clocks": clk,
                "replicas_identical": replicas_identical, "strong_scaling": strong, "other_configs": others,
                "ms_per_rank": ms_per_rank, "dp_mode": (arm.eng._dp_mode if world > 1 else "single")}
        emit(line)
    arm.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
