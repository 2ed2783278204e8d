"""The persistent LSTM scans row by row, against the float64 oracle (oracle/learner_oracle.py), at the batch sizes
where their tiling switches, at the chain lengths the learner runs, and with saturated gates.

The batch tiling of the scans depends on how many clusters the device keeps resident, so the batch sizes here are
derived from the device (r2d2_debug_max_active_clusters) and land on both sides of every switch:

  * pick_tiling (tcgen05, H <= 512): 16-row tiles while ceil(B/16) clusters fit, then 32-row tiles spread over the
    resident clusters, then several waves of full 32-row tiles;
  * the H = 512 forward kernel: ceil(B/resident) rows per cluster (at most 80), a cluster of more than 8 rows runs
    two sub-tiles of (n+1)/2 and n/2 rows, and the last cluster may have fewer rows than the others;
  * the H = 512 BPTT: full waves of 32-row clusters plus a second launch of 16-row clusters for the remainder;
  * pick_nb of the mma.sync kernels (H <= 256): 8, 16 or 32 rows per cluster for 148/(H/32) clusters.

Every comparison reports the worst ROW as well as the global relative L2 error: the error of row b,
||x[.., b, ..] - ref[.., b, ..]|| / (||ref|| / sqrt(B)), is measured against the RMS row norm, so a row that a
tile drops, misroutes or truncates shows up as an error of order 1 however large B is.  A failure names the row, the
cluster (and sub-tile) it belongs to, the step where its error peaks and the tensor.  Run with -s to see, for every
case, the tiling chosen and the errors measured.
"""
import ctypes
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, rel_l2
from oracle import learner_oracle as lo

pytestmark = pytest.mark.gpu

SMS = 148                 # B200 SM count: the mma.sync kernels size their tiles for 148 / (H/32) clusters
BIG_MAX_ROWS = 80         # rows per cluster of the H = 512 forward kernel


@pytest.fixture(scope="module")
def nv():
    from r2d2_b200 import native
    native.lib()
    return native


def dev(a):
    return torch.as_tensor(np.ascontiguousarray(a, dtype=np.float32)).cuda()


def f32(a):
    """The float32 value the kernel sees, as float64 for the oracle."""
    return np.asarray(a, np.float32).astype(np.float64)


def cdiv(a, b):
    return -(-a // b)


def env_on(name):
    e = os.environ.get(name)
    return not (e and e[0] == "0")


# ---------------------------------------------------------------------------------------------- tiling, as the library
# chooses it (lstm_scan_tc.cu: pick_tiling, fwd_big, bwd_tc; lstm_scan.cu: pick_nb)
def fits(nv, H):
    q = nv.lib().r2d2_debug_max_active_clusters
    d = {f"{k}{nb}{'b' if bwd else 'f'}": q(H, nb, bwd) for k, nb in (("fit", 16), ("fit", 32)) for bwd in (0, 1)}
    for k, v in list(d.items()):
        d[k] = v if v > 0 else SMS // (H // 32)
    big = q(512, 80, 0) if H == 512 else -1
    d["big"] = big if big > 0 else 7
    d["v1"] = SMS // (H // 32)
    return d


def pick_tiling(B, fit16, fit32):
    if cdiv(B, 16) <= fit16:
        return 16, 16, cdiv(B, 16)
    n = fit32
    if cdiv(B, n) > 32:
        n = cdiv(B, 32)
    rows = cdiv(B, n)
    return 32, rows, cdiv(B, rows)


def tiling(nv, H, B, backward, impl):
    """(description, clusters) of one scan call; clusters = [(first row, end row, label)] in launch order."""
    fd = fits(nv, H)
    if impl == 0:
        if H == 512:
            return "generic per-step GEMM path", [(0, B, "generic")]
        nb = next((o for o in (8, 16, 32) if cdiv(B, o) <= fd["v1"]), 32)
        return f"mma.sync {cdiv(B, nb)} x {nb} rows", [(c * nb, min(B, c * nb + nb), f"cluster {c}")
                                                       for c in range(cdiv(B, nb))]
    if H == 512 and not backward and env_on("R2D2_SCAN_L2XCHG"):
        rows = cdiv(B, fd["big"])
        if rows > BIG_MAX_ROWS:
            rows = cdiv(B, cdiv(B, BIG_MAX_ROWS))
        cl = []
        for c in range(cdiv(B, rows)):
            b0, b1 = c * rows, min(B, c * rows + rows)
            n = b1 - b0
            if n > 8:
                r0 = (n + 1) // 2
                cl += [(b0, b0 + r0, f"cluster {c} sub-tile 0 of {r0}"), (b0 + r0, b1, f"cluster {c} sub-tile 1 of {n - r0}")]
            else:
                cl.append((b0, b1, f"cluster {c} one sub-tile of {n}"))
        last = B - (cdiv(B, rows) - 1) * rows
        return (f"big fwd {cdiv(B, rows)} clusters x {rows} rows (last {last}), resident {fd['big']}, "
                f"{'mixed 1/2' if (last > 8) != (rows > 8) else ('two' if rows > 8 else 'one')} sub-tiles"), cl
    d = "b" if backward else "f"
    nb, rows, n = pick_tiling(B, fd[f"fit16{d}"], fd[f"fit32{d}"])
    kern = "tc" if not (H <= 256 and nb == 32 and not backward) else (
        "pingpong" if env_on("R2D2_SCAN_PINGPONG") else "tc")
    cl = [(c * rows, min(B, c * rows + rows), f"cluster {c}") for c in range(n)]
    desc = f"{kern} nb={nb}: {n} clusters x {rows} rows (last {B - (n - 1) * rows})"
    if H == 512 and backward and rows == 32 and env_on("R2D2_SCAN_L2XCHG"):
        fit = fd["fit32b"]
        full = (n // fit) * fit
        rest = B - full * 32
        if full > 0 and rest > 0 and cdiv(rest, 16) <= fit:
            cl = ([(c * 32, c * 32 + 32, f"launch 1 cluster {c}") for c in range(full)] +
                  [(full * 32 + c * 16, min(B, full * 32 + c * 16 + 16), f"launch 2 cluster {c}")
                   for c in range(cdiv(rest, 16))])
            desc = f"split BPTT: {full} x 32 rows + {cdiv(rest, 16)} x 16 rows"
    return desc, cl


def where(clusters, b):
    for b0, b1, label in clusters:
        if b0 <= b < b1:
            return f"{label}, rows [{b0},{b1})"
    return "no cluster"


# ---------------------------------------------------------------------------------------------- comparisons
def compare(name, x, ref, baxis, tol_g, tol_r, clusters=None):
    """Global relative L2 and worst-row error of x against ref (batch axis baxis; axis 0 is the step when baxis>0)."""
    x, ref = np.asarray(x, np.float64), np.asarray(ref, np.float64)
    B = ref.shape[baxis]
    dx, rr = np.moveaxis(x - ref, baxis, 0).reshape(B, -1), np.moveaxis(ref, baxis, 0).reshape(B, -1)
    nref = max(float(np.linalg.norm(rr)), 1e-30)
    rows = np.linalg.norm(dx, axis=1) / (nref / math.sqrt(B))
    b = int(np.nanargmax(rows)) if np.isfinite(rows).any() else 0
    if np.isnan(rows).any():
        b = int(np.argmax(np.isnan(rows)))
    rec = {"tensor": name, "global": float(np.linalg.norm(dx) / nref), "row": float(rows[b]), "b": b,
           "tol_g": tol_g, "tol_r": tol_r}
    if baxis > 0:
        per_step = np.linalg.norm(np.take(x - ref, b, axis=baxis).reshape(x.shape[0], -1), axis=1)
        rec["step"] = int(np.nanargmax(per_step)) if np.isfinite(per_step).any() else 0
    if clusters is not None:
        rec["where"] = where(clusters, b)
    return rec


def failures(recs):
    bad = []
    for r in recs:
        if not (r["global"] <= r["tol_g"] and r["row"] <= r["tol_r"]):
            bad.append(f"{r['tensor']}: worst row b={r['b']}" + (f" ({r['where']})" if "where" in r else "") +
                       (f" peaking at step {r['step']}" if "step" in r else "") +
                       f": row error {r['row']:.3e} (tol {r['tol_r']:.3g}), global {r['global']:.3e} "
                       f"(tol {r['tol_g']:.3g})")
    return bad


def show(head, recs):
    print(head)
    for r in recs:
        print(f"    {r['tensor']:<22} global {r['global']:.3e}  worst row {r['row']:.3e} (b={r['b']})")


def scan_status(nv):
    status = ctypes.c_int(0)
    nv.check(nv.lib().r2d2_scan_status(ctypes.byref(status), nv.current_stream()))
    return status.value


def head_rows(dh_head, S, B, H, repeat, first):
    """[S,B,H] head gradient as the scan consumes dh_head: row (s-first)/repeat at steps s >= first whose
    (s-first) % repeat == repeat-1 (lstm_scan.cuh, ScanBwdParams::dh_head)."""
    full = np.zeros((S, B, H))
    for s in range(first, S):
        if (s - first) % repeat == repeat - 1:
            full[s] = dh_head[(s - first) // repeat]
    return full


# ---------------------------------------------------------------------------------------------- 1. scan entry points
# (global, worst row), about 5x the worst values measured on a B200 (1000 W) over the whole sweep, both
# implementations: forward 1.0e-6 global / 1.8e-6 row (head_in), BPTT 1.4e-6 / 2.4e-6 (dgin)
SCAN_TOL = {"hs": (5e-6, 1e-5), "cs": (5e-6, 1e-5), "gates": (5e-6, 1e-5), "head_in": (5e-6, 1e-5),
            "dgates": (7e-6, 1.2e-5), "dgin": (7e-6, 1.2e-5)}

# variants of one batch size: (repeat, T, initial state given, gates alias gin, dgates alias gates, head_first_step)
VARIANTS = [(1, 6, True, True, True, 0), (2, 4, False, False, False, 3)]


def run_scan_case(nv, H, B, impl, seed, variants=VARIANTS, tol=SCAN_TOL):
    """Forward and BPTT of the scan entry points on scan implementation `impl`, each variant compared to
    learner_oracle.scan_forward / scan_backward.  Returns (tiling descriptions, records)."""
    lib = nv.lib()
    lib.r2d2_set_scan_impl(impl)
    recs, descs = [], []
    try:
        for vi, (repeat, T, with_state, alias_g, alias_dg, first) in enumerate(variants):
            rng = np.random.default_rng(seed * 10 + vi)
            S = T * repeat
            gin = f32(rng.standard_normal((T, B, 4 * H)))
            whh = f32(rng.uniform(-1, 1, (4 * H, H)) / math.sqrt(H))
            h0 = f32(rng.uniform(-0.9, 0.9, (B, H))) if with_state else np.zeros((B, H))
            c0 = f32(rng.standard_normal((B, H))) if with_state else np.zeros((B, H))
            g_ref, hs_ref, cs_ref = lo.scan_forward(gin, whh, h0, c0, repeat)
            head_ref = np.tanh(hs_ref[repeat::repeat])
            d_gin, d_whh = dev(gin), dev(whh)
            gates = d_gin if alias_g else torch.zeros((S, B, 4 * H), device="cuda")
            hs, cs = torch.zeros((S + 1, B, H), device="cuda"), torch.zeros((S + 1, B, H), device="cuda")
            head_in = torch.zeros((T, B, H), device="cuda")
            scratch = torch.zeros(B * 4 * H, device="cuda") if H == 512 else None
            d_h0, d_c0 = (dev(h0), dev(c0)) if with_state else (None, None)
            nv.check(lib.r2d2_lstm_scan_forward(nv.dptr(d_gin), nv.dptr(d_whh), nv.dptr(d_h0), nv.dptr(d_c0),
                                                nv.dptr(gates), nv.dptr(hs), nv.dptr(cs), nv.dptr(head_in), T, B, H,
                                                repeat, nv.dptr(scratch), nv.current_stream()))
            torch.cuda.synchronize()
            desc, cl = tiling(nv, H, B, False, impl)
            descs.append(f"fwd r{repeat}: {desc}")
            tag = f"r{repeat} "
            recs += [compare(tag + "hs", hs.cpu().numpy(), hs_ref, 1, *tol["hs"], cl),
                     compare(tag + "cs", cs.cpu().numpy(), cs_ref, 1, *tol["cs"], cl),
                     compare(tag + "gates", gates.cpu().numpy(), g_ref, 1, *tol["gates"], cl),
                     compare(tag + "head_in", head_in.cpu().numpy(), head_ref, 1, *tol["head_in"], cl)]
            # BPTT from the oracle's saved activations (as float32), so that forward errors do not enter it
            g32, hs32, cs32 = f32(g_ref), f32(hs_ref), f32(cs_ref)
            n_head = (S - first) // repeat
            dh_head = f32(rng.standard_normal((n_head, B, H)))
            dg_ref, _, _ = lo.scan_backward(g32, cs32, whh, head_rows(dh_head, S, B, H, repeat, first))
            dgin_ref = dg_ref.reshape(T, repeat, B, 4 * H).sum(1)
            d_g = dev(g32)
            dgates = d_g if alias_dg else torch.zeros((S, B, 4 * H), device="cuda")
            dgin = torch.zeros((T, B, 4 * H), device="cuda") if repeat > 1 else None
            bscratch = torch.zeros(2 * B * H, device="cuda") if H == 512 else None
            d_hs, d_cs, d_dh = dev(hs32), dev(cs32), dev(dh_head)
            nv.check(lib.r2d2_lstm_scan_backward(nv.dptr(d_g), nv.dptr(d_hs), nv.dptr(d_cs), nv.dptr(d_whh),
                                                 nv.dptr(d_dh), first, nv.dptr(dgates), nv.dptr(dgin), T, B, H, repeat,
                                                 nv.dptr(bscratch), nv.current_stream()))
            torch.cuda.synchronize()
            desc, cl = tiling(nv, H, B, True, impl)
            descs.append(f"bwd r{repeat}: {desc}")
            recs.append(compare(tag + "dgates", dgates.cpu().numpy(), dg_ref, 1, *tol["dgates"], cl))
            if repeat > 1:
                recs.append(compare(tag + "dgin", dgin.cpu().numpy(), dgin_ref, 1, *tol["dgin"], cl))
    finally:
        lib.r2d2_set_scan_impl(1)
    return descs, recs


# batch sizes, as formulas of the device's resident-cluster counts (fits()): the two sides of every tiling switch
B_COMMON = ["1", "16*fit16f", "16*fit16f+1", "16*fit16b", "16*fit16b+1", "32*fit32f", "32*fit32f+1",
            "32*fit32b", "32*fit32b+1"]
B_V1 = ["8*v1", "8*v1+1", "16*v1", "16*v1+1"]
B_512 = ["8*big", "8*big+1", "80*big", "80*big+1", "480", "512"]


def b_labels(H):
    return B_COMMON + (B_512 if H == 512 else B_V1)


def resolve(label, fd):
    return int(eval(label, {}, dict(fd)))   # labels are the fixed formulas above


SCAN_CASES = [(H, lab) for H in (32, 64, 128, 256, 512) for lab in b_labels(H)]


@pytest.mark.parametrize("impl", [1, 0], ids=["tc", "mma"])
@pytest.mark.parametrize("H,label", SCAN_CASES)
def test_scan_tiling_sweep(nv, H, label, impl):
    B = resolve(label, fits(nv, H))
    descs, recs = run_scan_case(nv, H, B, impl, seed=H * 7919 + B)
    show(f"scan H={H} B={B} ({label}) impl={'tc' if impl else 'mma'}\n    " + "\n    ".join(descs), recs)
    assert scan_status(nv) == 0, "a bounded mbarrier wait timed out inside a scan kernel"
    bad = failures(recs)
    assert not bad, f"H={H} B={B} ({label}) impl={impl}:\n" + "\n".join(bad)


# ---------------------------------------------------------------------------------------------- net entry points
def make_params(rng, O, A, H, critic):
    I = O + (A if critic else 0)
    u = lambda shp, b: rng.uniform(-b, b, shp)  # noqa: E731
    return {"l1.weight": u((H, I), 1 / np.sqrt(H)), "l1.bias": u((H,), 0.2),
            "l2.weight_ih": u((4 * H, H), 1 / np.sqrt(H)), "l2.weight_hh": u((4 * H, H), 1 / np.sqrt(H)),
            "l2.bias_ih": u((4 * H,), 0.1), "l2.bias_hh": u((4 * H,), 0.1),
            "l3.weight": u((A, H), 0.1), "l3.bias": u((A,), 0.1)}


def run_net(nv, O, A, H, B, T, repeat, critic, first_row, seed, tol, fp32_scale=False):
    """r2d2_lstm_net_forward / _backward (tcgen05 scan: operand images, fused bias sums) against the float64
    oracle.  Per row: out and d_act; globally: the eight gradient blocks."""
    rng = np.random.default_rng(seed)
    p = {k: f32(v) for k, v in make_params(rng, O, A, H, critic).items()}
    obs, act = f32(rng.standard_normal((T, B, O))), f32(rng.uniform(-1, 1, (T, B, A)))
    h0, c0 = f32(0.3 * rng.standard_normal((B, H))), f32(0.3 * rng.standard_normal((B, H)))
    x = np.concatenate((obs, act), 2) if critic else obs
    d_out_rows = f32(rng.standard_normal((T - first_row, B, A)))

    def oracle(dt):
        cv = lambda a: np.asarray(a, dt)  # noqa: E731
        sv = lo.net_forward({k: cv(v) for k, v in p.items()}, cv(x), cv(h0), cv(c0), critic=critic, repeat=repeat)
        d_full = np.zeros_like(sv["out"])
        d_full[repeat - 1::repeat][first_row:] = d_out_rows
        g, dx, _ = lo.net_backward({k: cv(v) for k, v in p.items()}, sv, d_full, critic=critic, want_wgrad=True,
                                   want_dx=critic)
        return sv["out"][repeat - 1::repeat][first_row:], g, (dx[:, :, O:] if critic else None)

    out_ref, g_ref, dact_ref = oracle(np.float64)
    lib = nv.lib()
    shape = nv.NetShape(O, A, H, int(critic))
    ws = torch.zeros(lib.r2d2_net_workspace_floats(nv.byref(shape), T, B, repeat), device="cuda")
    flat = np.concatenate([p[k].reshape(-1) for k in lo.PARAM_KEYS])
    dparams, dobs, dact, dh0, dc0 = dev(flat), dev(obs), dev(act), dev(h0), dev(c0)
    out = torch.zeros((T - first_row, B, A), device="cuda")
    nv.check(lib.r2d2_lstm_net_forward(nv.byref(shape), nv.dptr(dparams), nv.dptr(dobs), nv.dptr(dact) if critic else None,
                                       nv.dptr(dh0), nv.dptr(dc0), T, B, repeat, first_row, nv.dptr(out), nv.dptr(ws),
                                       nv.current_stream()))
    grads = torch.zeros(flat.size, device="cuda")
    d_act = torch.zeros((T, B, A), device="cuda") if critic else None
    d_out = dev(d_out_rows)
    nv.check(lib.r2d2_lstm_net_backward(nv.byref(shape), nv.dptr(dparams), nv.dptr(dobs),
                                        nv.dptr(dact) if critic else None, nv.dptr(d_out), T, B, repeat, first_row,
                                        nv.dptr(grads), nv.dptr(d_act), nv.dptr(ws), nv.current_stream()))
    torch.cuda.synchronize()
    _, cl = tiling(nv, H, B, True, nv.lib().r2d2_get_scan_impl())
    recs = [compare("out", out.cpu().numpy(), out_ref, 1, *tol["out"], cl)]
    g = grads.cpu().numpy()
    off = 0
    for k in lo.PARAM_KEYS:
        n = g_ref[k].size
        recs.append(compare(f"grad {k}", g[off:off + n].reshape(1, -1), g_ref[k].reshape(1, -1), 0, *tol["grad"]))
        off += n
    if critic:
        recs.append(compare("d_act", d_act.cpu().numpy(), dact_ref, 1, *tol["d_act"], cl))
    if fp32_scale:   # the same computation in float32 on the CPU, for scale
        o32, g32, a32 = oracle(np.float32)
        scale = {"out": rel_l2(o32, out_ref), "grads": max(rel_l2(g32[k], g_ref[k]) for k in lo.PARAM_KEYS)}
        if critic:
            scale["d_act"] = rel_l2(a32, dact_ref)
        print("    fp32 CPU oracle vs float64: " + ", ".join(f"{k} {v:.3e}" for k, v in scale.items()))
    return recs


# measured on a B200: out 3.5e-6 / 6.9e-6 row, gradients 8.7e-6, d_act 8.2e-6 / 1.8e-5 row
NET_TOL = {"out": (2e-5, 3.5e-5), "grad": (4.5e-5, 4.5e-5), "d_act": (4e-5, 9e-5)}
NET_CASES = [(H, lab) for H in (32, 64, 128, 256, 512) for lab in b_labels(H)]


@pytest.mark.parametrize("H,label", NET_CASES)
def test_net_critic_tiling_sweep(nv, H, label):
    """Critic net (operand-image BPTT path, fused bias sums) at the batch sizes of the scan sweep."""
    B = resolve(label, fits(nv, H))
    recs = run_net(nv, 20, 4, H, B, 5, 1, True, 1, seed=H * 31 + B, tol=NET_TOL)
    show(f"critic net H={H} B={B} ({label})\n    fwd: {tiling(nv, H, B, False, 1)[0]}\n    "
         f"bwd: {tiling(nv, H, B, True, 1)[0]}", recs)
    assert scan_status(nv) == 0, "a bounded mbarrier wait timed out inside a scan kernel"
    bad = failures(recs)
    assert not bad, f"critic net H={H} B={B} ({label}):\n" + "\n".join(bad)


# ---------------------------------------------------------------------------------------------- 3. full chain length
# production window sizes: critic T = 125 rows with head outputs from row 40, actor T = 80 rows x 2 cell steps.
# Tolerances: 5x the worst values measured on a B200 (see the docstring of test_full_chain).
CHAIN_TOL = {"out": (1.75e-5, 2.1e-5), "grad": (1.45e-4, 1.45e-4), "d_act": (3.3e-5, 4e-5)}


@pytest.mark.parametrize("kind", ["critic", "actor"])
@pytest.mark.parametrize("H,B", [(256, 256), (256, 257), (512, 24), (512, 512)])
def test_full_chain(nv, H, B, kind):
    """Net entry points at the learner's chain lengths against float64 (obs 20, act 4: the scan is under test).

    Worst values measured on a B200 (1000 W) over the eight cases, which the tolerances are 5x of: out 3.5e-6 global,
    4.2e-6 worst row; gradients 2.9e-5 (l2.weight_hh of the actor chain at H = 512, B = 512; 6.8e-6 or less at the
    other shapes); d_act 6.6e-6 global, 8.0e-6 worst row.  The same computation in float32 on the CPU is off the
    float64 result by 1.6e-7 .. 2.9e-7 (out), 7.9e-7 .. 5.6e-6 (gradients), 3.2e-7 .. 4.7e-7 (d_act)."""
    critic = kind == "critic"
    T, repeat, first = (125, 1, 40) if critic else (80, 2, 0)
    print(f"\n{kind} chain H={H} B={B} T={T} repeat={repeat}\n    fwd: {tiling(nv, H, B, False, 1)[0]}\n    "
          f"bwd: {tiling(nv, H, B, True, 1)[0]}")
    recs = run_net(nv, 20, 4, H, B, T, repeat, critic, first, seed=H + B + repeat, tol=CHAIN_TOL, fp32_scale=True)
    show("   ", recs)
    assert scan_status(nv) == 0, "a bounded mbarrier wait timed out inside a scan kernel"
    bad = failures(recs)
    assert not bad, f"{kind} chain H={H} B={B}:\n" + "\n".join(bad)


# ---------------------------------------------------------------------------------------------- 4. saturation
LOG2E = 1.4426950408889634
SIG_EDGE = 43 / LOG2E          # sigmoid_pair clamps the exponent at 43: sigma(x) for x < -SIG_EDGE
TANH_EDGE = 43 / (2 * LOG2E)   # tanh(x) = 2 sigma(2x) - 1 (g gate, tanh(c))
ULPS = (-4, -2, -1, 0, 1, 2, 4)


def edge(v, k):
    """v moved by k float32 ulps."""
    x = np.float32(v)
    for _ in range(abs(k)):
        x = np.nextafter(x, np.float32(np.inf if k > 0 else -np.inf), dtype=np.float32)
    return float(x)


def saturated_inputs(H, B, T, seed):
    """gin [T,B,4H], whh, c0 with: pre-activations over [-60, 60]; sigma / tanh arguments at the clamp edge +- a few
    ulp; exact zeros; f = i = 1, g = +-1 so that |c| grows by 1 per step from c0 = +-30; c parked at +-TANH_EDGE.
    The W_hh rows of those units are zero, so the kernel's pre-activation is exactly the chosen gin."""
    rng = np.random.default_rng(seed)
    gin = rng.uniform(-60, 60, (T, B, 4 * H))
    small = rng.uniform(size=(T, B, 4 * H)) < 0.3
    gin[small] = rng.standard_normal(int(small.sum()))
    whh = rng.uniform(-1, 1, (4 * H, H)) / math.sqrt(H)
    c0 = np.where(rng.uniform(size=(B, H)) < 0.5, 30.0, -30.0)
    c0[:, H // 2:] = rng.standard_normal((B, H - H // 2))
    units = rng.permutation(H)
    u_edge, u_grow, u_zero, u_cedge = units[:16], units[16:24], units[24:28], units[28:36]
    for q in range(4):
        whh[q * H + np.concatenate((u_edge, u_grow, u_zero, u_cedge))] = 0
    t_, b_ = np.meshgrid(np.arange(T), np.arange(B), indexing="ij")
    for j, u in enumerate(u_edge):
        k = np.vectorize(lambda i: ULPS[i % len(ULPS)])(t_ + b_ + j)
        sgn = np.where(((t_ + j) // 7) % 2 == 0, -1.0, 1.0)
        for q in range(4):
            base = TANH_EDGE if q == 2 else SIG_EDGE
            gin[:, :, q * H + u] = sgn * np.vectorize(edge)(base, k)
    for j, u in enumerate(u_grow):   # i = f = 1, g = +-1: c_s = c0 +- s
        gin[:, :, u], gin[:, :, H + u] = 40.0, 40.0
        gin[:, :, 2 * H + u] = np.where((b_ + j) % 2 == 0, 40.0, -40.0)
    gin[:, :, np.concatenate([q * H + u_zero for q in range(4)])] = 0.0
    c0[:, u_zero] = 0.0
    for j, u in enumerate(u_cedge):  # i = 0, f = 1, g = 0: c stays at c0 = +-TANH_EDGE +- ulps for every step
        gin[:, :, u], gin[:, :, H + u], gin[:, :, 2 * H + u] = -60.0, 60.0, 0.0
        c0[:, u] = [(1 if (b + j) % 2 else -1) * edge(TANH_EDGE, ULPS[(b + j) % len(ULPS)]) for b in range(B)]
    return f32(gin), f32(whh), f32(c0)


# absolute error of hs / gates (relative error is ill-posed at 0 and 1); cs relative to 1 + |c|; dgates relative to
# ||dh_head||.  About 5x the worst values measured on a B200: hs 7.9e-6, gates 5.1e-6, cs 7.1e-6 (at |x| <= 60 one
# float32 ulp of the pre-activation is up to 3.8e-6), dgates 1.1e-7 global and worst row.  A sigmoid that stops at
# 2^-8 instead of ~0 below x = -5.5 is off by 3.9e-3.
SAT_TOL = {"hs": 4e-5, "gates": 2.5e-5, "cs": 3.5e-5, "dgates": (5.5e-7, 5.5e-7)}


@pytest.mark.parametrize("tile", ["16-row", "32-row"])
@pytest.mark.parametrize("H", [128, 256, 512])
def test_saturated_gates(nv, H, tile):
    T = 125
    fd = fits(nv, H)
    B = 16 if tile == "16-row" else 16 * max(fd["fit16f"], fd["fit16b"]) + 1
    gin, whh, c0 = saturated_inputs(H, B, T, seed=H + B)
    h0 = np.zeros((B, H))
    g_ref, hs_ref, cs_ref = lo.scan_forward(gin, whh, h0, c0, 1)
    lib = nv.lib()
    d_gin, d_whh, d_c0 = dev(gin), dev(whh), dev(c0)
    gates = torch.zeros((T, B, 4 * H), device="cuda")
    hs, cs = torch.zeros((T + 1, B, H), device="cuda"), torch.zeros((T + 1, B, H), device="cuda")
    head_in = torch.zeros((T, B, H), device="cuda")
    nv.check(lib.r2d2_lstm_scan_forward(nv.dptr(d_gin), nv.dptr(d_whh), None, nv.dptr(d_c0), nv.dptr(gates),
                                        nv.dptr(hs), nv.dptr(cs), nv.dptr(head_in), T, B, H, 1, None,
                                        nv.current_stream()))
    rng = np.random.default_rng(H)
    dh_head = f32(rng.standard_normal((T, B, H)))
    g32, cs32 = f32(g_ref), f32(cs_ref)
    dg_ref, _, _ = lo.scan_backward(g32, cs32, whh, dh_head)
    d_g, d_cs, d_hs, d_dh = dev(g32), dev(cs32), dev(f32(hs_ref)), dev(dh_head)
    dgates = torch.zeros((T, B, 4 * H), device="cuda")
    nv.check(lib.r2d2_lstm_scan_backward(nv.dptr(d_g), nv.dptr(d_hs), nv.dptr(d_cs), nv.dptr(d_whh), nv.dptr(d_dh), 0,
                                         nv.dptr(dgates), None, T, B, H, 1, None, nv.current_stream()))
    torch.cuda.synchronize()
    assert scan_status(nv) == 0, "a bounded mbarrier wait timed out inside a scan kernel"
    out = {"hs": hs.cpu().numpy(), "cs": cs.cpu().numpy(), "gates": gates.cpu().numpy(),
           "head_in": head_in.cpu().numpy(), "dgates": dgates.cpu().numpy()}
    for k, v in out.items():
        assert np.isfinite(v).all(), f"H={H} B={B}: non-finite {k} at {np.argwhere(~np.isfinite(v))[:4].tolist()}"
    _, clf = tiling(nv, H, B, False, 1)
    _, clb = tiling(nv, H, B, True, 1)
    bad, lines = [], []
    for k, ref, scale in (("hs", hs_ref, 0.0), ("gates", g_ref, 0.0), ("cs", cs_ref, 1.0)):
        err = np.abs(out[k] - ref) / (1.0 + np.abs(ref)) if scale else np.abs(out[k] - ref)
        s, b, e = np.unravel_index(int(np.argmax(err)), err.shape)
        what = f"gate {e // H} unit {e % H}" if k == "gates" else f"unit {e}"
        lines.append(f"{k} max abs err {err.max():.3e} at step {s} row b={b} {what} (ref {ref[s, b, e]:.6g}, "
                     f"x = {gin[min(s, T - 1), b, e] if k == 'gates' else cs_ref[s, b, e]:.9g})")
        if not err.max() <= SAT_TOL[k]:
            bad.append(lines[-1] + f" > {SAT_TOL[k]:.3g} ({where(clf, b)})")
    # dgates: error relative to ||dh_head||, globally and per row
    d = (out["dgates"] - dg_ref).transpose(1, 0, 2).reshape(B, -1)
    nh = float(np.linalg.norm(dh_head))
    rows = np.linalg.norm(d, axis=1) / (nh / math.sqrt(B))
    b = int(np.argmax(rows))
    gl = float(np.linalg.norm(d)) / nh
    lines.append(f"dgates err / ||dh_head|| global {gl:.3e} worst row {rows[b]:.3e} (b={b})")
    if not (gl <= SAT_TOL["dgates"][0] and rows[b] <= SAT_TOL["dgates"][1]):
        bad.append(lines[-1] + f" ({where(clb, b)})")
    print(f"\nsaturated H={H} B={B} S={T}\n    fwd: {tiling(nv, H, B, False, 1)[0]}\n    bwd: "
          f"{tiling(nv, H, B, True, 1)[0]}\n    " + "\n    ".join(lines))
    assert not bad, f"saturated H={H} B={B}:\n" + "\n".join(bad)


# ---------------------------------------------------------------------------------------------- 5. engine vs float64
# per (t, b) for q / target / td_sq, per b for the priority; losses, gradients and post-Adam weights globally
# measured on a B200: q 4.8e-6 / 5.6e-6 row, target 1.1e-7 / 1.2e-7, td_sq 1.3e-7 / 1.8e-7, priority 1.0e-7 / 2.9e-7,
# losses 8.7e-6, gradients 1.6e-5, post-Adam weights 2.9e-5 (l3.weight: Adam's first step moves every element by about
# lr whatever its gradient, so the relative error of small gradients carries over).  Split-K sums run in atomic order,
# hence about 10x on the smallest ones.
ENGINE_TOL = {"q": (2.5e-5, 3e-5), "target": (1e-6, 1.2e-6), "td_sq": (1e-6, 1.5e-6), "priority": (1e-6, 2e-6),
              "loss": 5e-5, "grad": 8e-5, "after": 1.5e-4}


@pytest.mark.parametrize("B", [57, 113])
def test_engine_against_float64_learner(nv, B):
    """LearnerEngine at H = 512 (burn-in 40, learning 80, n = 5) against OracleLearner in float64, two iterations.
    B = 57: one forward launch mixes clusters with one and two sub-tiles; B = 113: the BPTT runs 17-row clusters on
    32-row tiles.  target_q_value is where the inference-only target chains are observable."""
    from oracle import ref_port
    from r2d2_b200 import engine
    cfg = engine.PathConfig(obs=20, act=4, hidden=512, batch=B, burn_in=40, learning=80, n_step=5)
    pc = ref_port.PathConfig(obs=20, act=4, hidden=512, batch=B, burn_in=40, learning=80, n_step=5)
    eng = engine.LearnerEngine(cfg, seed=5)
    init = {n: {k: v.cpu().numpy() for k, v in eng.views(n).items()} for n in ("actor", "critic")}
    ol = lo.OracleLearner(init["actor"], init["critic"], burn_in=40, learning=80, n_step=5)
    L = cfg.learning
    for it in range(2):
        batch = ref_port.synthetic_batch(pc, seed=10 + it)
        ref = ol.iteration(batch)
        eng.set_batch(batch)
        eng.step()
        torch.cuda.synchronize()
        assert scan_status(nv) == 0, "a bounded mbarrier wait timed out inside a scan kernel"
        _, cl = tiling(nv, 512, B, False, 1)
        recs = [compare("q_value", eng.q_value.cpu().numpy().reshape(L, B, -1), ref["q_value"].reshape(L, B, -1), 1,
                        *ENGINE_TOL["q"], cl),
                compare("target_q_value", eng.target_q_value.cpu().numpy().reshape(L, B, -1),
                        ref["target_q_value"].reshape(L, B, -1), 1, *ENGINE_TOL["target"], cl),
                compare("td_sq", eng.td_sq.cpu().numpy().reshape(L, B), ref["average_td_loss"].reshape(L, B), 1,
                        *ENGINE_TOL["td_sq"], cl),
                compare("priority", eng.priority.cpu().numpy(), ref["priority"], 0, *ENGINE_TOL["priority"], cl)]
        losses = eng.losses.cpu().numpy()
        for i, k in enumerate(("critic_loss", "actor_loss")):
            e = abs(float(losses[i]) - ref[k]) / max(abs(ref[k]), 1e-12)
            recs.append({"tensor": k, "global": e, "row": e, "b": 0, "tol_g": ENGINE_TOL["loss"],
                         "tol_r": ENGINE_TOL["loss"]})
        for net in ("actor", "critic"):
            gr = {k: v.cpu().numpy() for k, v in eng.views(net, "grads").items()}
            pa = {k: v.cpu().numpy() for k, v in eng.views(net).items()}
            for k in lo.PARAM_KEYS:
                for what, a, r, tl in (("grad", gr[k], ref[f"{net}_grad"][k], ENGINE_TOL["grad"]),
                                       ("after", pa[k], ref[f"{net}_after"][k], ENGINE_TOL["after"])):
                    e = rel_l2(a, r)
                    recs.append({"tensor": f"{net}_{what}/{k}", "global": e, "row": e, "b": 0, "tol_g": tl, "tol_r": tl})
        print(f"\nengine H=512 B={B} iteration {it}\n    fwd: {tiling(nv, 512, B, False, 1)[0]}\n    "
              f"bwd: {tiling(nv, 512, B, True, 1)[0]}")
        show("   ", recs)
        bad = failures(recs)
        assert not bad, f"engine B={B} iteration {it}:\n" + "\n".join(bad)


# ---------------------------------------------------------------------------------------------- 6. fallback kernels
def fallback_cases():
    """(H, batch label) rows the A/B kernels take: the H = 512 rows of the sweep and the 32-row tiles of H <= 256."""
    rows = [(512, lab) for lab in b_labels(512)]
    rows += [(H, lab) for H in (32, 64, 128, 256) for lab in ("16*fit16f+1", "32*fit32f", "32*fit32f+1")]
    return rows


@pytest.mark.parametrize("switch", ["R2D2_SCAN_L2XCHG", "R2D2_SCAN_PINGPONG"])
def test_fallback_kernels(switch):
    """The A/B kernels read their switch once per process: run the sweep's rows in a fresh interpreter
    (tests/scan_edges_worker.py) with the switch off and check the worst errors it reports."""
    env = dict(os.environ, **{switch: "0"})
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.join(ROOT, "tests",
                                                                                       "scan_edges_worker.py")]
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, f"worker failed ({r.returncode}):\n{r.stdout[-3000:]}\n{r.stderr[-3000:]}"
    res = json.loads(r.stdout.strip().splitlines()[-1])
    bad = []
    for c in res["cases"]:
        print(f"{switch}=0 H={c['H']} B={c['B']} ({c['label']}): " + "; ".join(c["tiling"]) +
              f"; worst global {max(x['global'] for x in c['records']):.3e} row "
              f"{max(x['row'] for x in c['records']):.3e}")
        bad += [f"H={c['H']} B={c['B']}: {m}" for m in failures(c["records"])]
    assert res["status"] == 0, "a bounded mbarrier wait timed out inside a scan kernel"
    assert len(res["cases"]) == len(fallback_cases())
    assert not bad, "\n".join(bad)
