#!/usr/bin/env python
"""bench.py -- BPR train triples/s (+ top-K users/s) of the Recommender hot path.

  python bench.py --gpus N --steps K --warmup W            # our CUDA path
  python bench.py --impl reference --gpus N --steps K ...  # CPU arm (oracle port, all host cores)
  python bench.py --steps K --dump-outputs DIR             # + what the last timed step computed, as DIR/*.npy

Workload (BASELINE.json configs[1]): 1M users / 200k recipes / 95 labels, D=128, BPR
triples (uniform users, Zipf(1.05) positives, uniform negatives), Adam with TF-1.x
semantics (lazy-exact), global-norm clip 5.0, General_Memory write every step.
One step = one fr_train_step over B triples.  Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CFG2 = dict(U=1_000_000, I=200_000, L=95, D=128)
CFG3 = dict(U=100_000_000, I=10_000_000, L=95, D=128)   # BASELINE configs[2]: needs the 8-GPU row-sharded path
SMALL = dict(U=20_000, I=5_000, L=95, D=128)       # --small: functional check of the harness only
METRIC, UNIT = "bpr_train_triples_per_sec", "triples/s"


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of each kernel, from the `ncu --set full` captures of THIS
    build's bench command (profiles/summarize.py traffic -> profiles/ncu_traffic.json: {"build": source hash,
    "kernels": {name: {"dram_bytes": ..., "capture": file}}}).  Returned only when the file was made from the sources
    the loaded library was built from; otherwise every `traffic` field in the line is null (nothing is hard-coded)."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(p):
        return {}
    try:
        j = json.load(open(p))
        from foodrec_b200 import _build
        if j.get("build") != _build.source_hash():
            return {}
        return {k: v["dram_bytes"] for k, v in j.get("kernels", {}).items()}
    except Exception:
        return {}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def tensor_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return float(j["bf16_tflops"]), float(j["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json bf16_tflops burst / sustained)"
    return 1590.0, 1400.0, "fallback (B200_PROFILING.md 1.59 PFLOP/s burst, ~1.4 sustained)"


def bench_catalog(eng, dev, label, n_users, K=100, reps=2, warm_users=None):
    """Full-catalog top-K users/s (fr_catalog_topk): device-timed with resident inputs, per-phase CUDA
    events from inside the library, and end to end from a pinned host user list to host ids."""
    import torch
    eng.catalog_prepare()
    info = eng.catalog_info()
    tile_n, sets, split = info["epi_sets"] % 1000, info["epi_sets"] // 1000, info["cta_group"] >= 10
    eng.timing_enable(True)
    eng.catalog_topk(n_users=warm_users or n_users, K=K)           # warm-up (workspace allocation, code load)
    torch.cuda.synchronize(); eng.catalog_timing_read()
    best = None
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); ids, sc = eng.catalog_topk(n_users=n_users, K=K); e1.record(); torch.cuda.synchronize()
        ph, passes = eng.catalog_timing_read()
        ms = e0.elapsed_time(e1)
        if best is None or ms < best[0]:
            best = (ms, ph, passes)
    ms, ph, passes = best
    fallback = eng.catalog_fallback_rows()
    eng.timing_enable(False)
    # e2e: pinned host user ids -> device, top-K, ids back to pinned host memory
    hu = torch.arange(n_users, dtype=torch.int32).pin_memory()
    hout = torch.empty((n_users, K), dtype=torch.int32).pin_memory()
    du = torch.empty(n_users, dtype=torch.int32, device=dev)
    torch.cuda.synchronize(); t0 = time.perf_counter()
    du.copy_(hu, non_blocking=True)
    ids = eng.catalog_topk(users=du, K=K, return_scores=False)
    hout.copy_(ids, non_blocking=True)
    torch.cuda.synchronize(); dt = time.perf_counter() - t0
    burst, sustained, src = tensor_peaks()
    executed = 2.0 * n_users * info["tiles"] * tile_n * info["k_padded"] * (2 if split else 1)
    dense = 2.0 * n_users * eng.I * 5 * eng.D                     # SURVEY 8(d): the K=5D contraction this replaces
    gemm_s = ph["gemm_filter"] * 1e-3
    return {
        "metric": "catalog_topk_users_per_sec", "workload": label, "value": n_users / (ms * 1e-3), "unit": "users/s",
        "users": n_users, "recipes": eng.I, "K": K, "ms": ms, "passes": passes, "phases_ms": ph, "fallback_rows": fallback,
        "kernel": {"cta_group": info["cta_group"] % 10, "epilogue_sets": sets, "tile_n": tile_n, "k_padded": info["k_padded"],
                   "split_user_operand": bool(split), "tiles": info["tiles"]},
        "roofline": {"bound": "tensor", "kernel": "catalog_gemm_kernel", "achieved": executed / gemm_s / 1e12, "peak": sustained,
                     "unit": "TFLOP/s", "frac": executed / gemm_s / 1e12 / sustained, "peak_burst": burst, "peak_source": src,
                     "traffic": ncu_traffic().get("catalog_gemm_kernel:" + label.split(":")[0]),
                     "flop_executed_total": executed, "gemm_ms_total": ph["gemm_filter"], "launches": passes,
                     "flop_per_launch_executed": executed / max(passes, 1), "ms_per_launch": ph["gemm_filter"] / max(passes, 1),
                     "dense_equivalent_tflops": dense / gemm_s / 1e12,
                     "note": "executed = bf16 MMA flops issued (mask-grouped K=D contraction, x2 for the split user operand); "
                             "dense_equivalent = SURVEY 8(d)'s 2*U*I*5D over the same time"},
        "e2e": {"value": n_users / dt, "unit": "users/s", "h2d_bytes": 4 * n_users, "d2h_bytes": 4 * n_users * K,
                "feed": "user ids from pinned host memory, top-K ids back to pinned host memory"},
    }


def bind_to_gpu_numa_node(index):
    """Run this process (and so first-touch its pinned feed buffers) on the CPU socket the GPU hangs off: the e2e
    number is an H2D copy of 111 MB per step, and a process that lands on the far socket copies across the
    inter-socket link (measured 68 vs 122 M triples/s on different boxes of the same pool).  Returns what it did;
    the CPU legs restore the full affinity first."""
    info = {"bound": False}
    try:
        bus = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(index)],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        if bus.count(":") == 2 and len(bus.split(":")[0]) == 8:
            bus = bus[4:]                                   # 00000000:1B:00.0 -> 0000:1b:00.0
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        info.update(pci=bus, numa_node=node)
        if node < 0:
            return info
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0)
        use = cpus & allowed
        info.update(node_cpus=len(cpus), allowed=len(allowed), used=len(use))
        if use and use != allowed:
            os.sched_setaffinity(0, use)
            info["bound"] = True
    except Exception as e:                                  # sysfs not exposed in this container: leave it alone
        info["error"] = type(e).__name__
    return info


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index
        self.t0 = self.t1 = None

    def start(self):
        """Started before the warm-up (nvidia-smi needs ~0.5 s to produce its first line);
        mark_begin/mark_end bracket the timed region."""
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "20"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self):
        if self.proc:
            self.proc.terminate()
        ok = lambda r: len(r) >= 7 and r[0].replace(".", "").isdigit()
        inside = [r for t, r in self.rows if ok(r) and self.t0 is not None and self.t0 <= t <= self.t1 + 0.02]
        window = "timed region"
        if len(inside) < 3:      # region shorter than the sampling period: use the whole loaded span
            lo = (self.t0 or 0) - 1.0
            inside = [r for t, r in self.rows if ok(r) and lo <= t <= (self.t1 or 1e18) + 0.05] or \
                     [r for _, r in self.rows if ok(r)]
            window = "pre-roll + warm-up + timed region (the 1 s up to the end of the timed region)"
        sm = [float(r[0]) for r in inside]
        mx = [float(r[1]) for r in inside]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(r[3 + k] == "Active" for r in inside)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max((float(r[2]) for r in inside), default=None),
                "samples": len(sm), "window": window, "reasons": reasons}


def make_batches(cfg, B, nb, seed, item_cats, lab_csr, dense):
    """nb BPR batches: ids only, plus (dense) the reference-format feed tensors."""
    import synth_data as synth
    out = []
    for k in range(nb):
        rng = np.random.default_rng(seed + k)
        users = rng.integers(0, cfg["U"], B).astype(np.int32)
        pos = synth.zipf_items(rng, cfg["I"], B)
        neg = rng.integers(0, cfg["I"], B).astype(np.int32)
        neg[neg == pos] = (neg[neg == pos] + 1) % cfg["I"]
        items = np.stack([pos, neg], 1).reshape(-1).copy()
        b = dict(users=users, items=items)
        if dense:
            b["cats"] = item_cats[items].copy()                                   # [2B,4]  categories
            b["ulab"] = synth.csr_rows_dense(lab_csr[0], lab_csr[1], users, cfg["L"])   # [B,L] user_one_hot_label
        out.append(b)
    return out


# ----------------------------------------------------------------------------- CPU arm
def run_reference(args, cfg, B):
    """The reference's CPU implementation of the path = the oracle's torch-CPU port
    (TensorFlow 1.x cannot be installed here: oracle/cpu_port.py header), on all host
    cores, on a bounded sample: `steps` BPR steps of B triples at the same table sizes."""
    import torch
    import synth_data as synth
    from oracle.cpu_port import CpuPort
    from oracle.recommender_oracle import Hyper
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = len(os.sched_getaffinity(0))
    torch.set_num_threads(cores)
    g = torch.Generator().manual_seed(1)
    U, I, L, D = cfg["U"], cfg["I"], cfg["L"], cfg["D"]
    P = torch.randn((U, 5, D), generator=g) * 0.1; R = torch.randn((I, D), generator=g) * 0.1
    Cat = torch.randn((4, D), generator=g) * 0.1; G = torch.randn((L, 5, D), generator=g) * 0.1
    item_cats = synth.make_item_categories(I)
    lab = synth.make_user_label_csr(U, L)
    port = CpuPort(P, R, Cat, G, Hyper(learner="adam", lr=0.001), threads=cores)
    del P
    steps, warm = args.steps, max(1, min(args.warmup, 1))
    bs = make_batches(cfg, B, steps + warm, 777, item_cats, lab, dense=True)
    T = lambda x, dt=None: torch.as_tensor(x if dt is None else x.astype(dt))
    t0 = None
    for k, b in enumerate(bs):
        if k == warm:
            t0 = time.perf_counter()
        it = T(b["items"], np.int64)
        port.train_step_bpr(T(b["users"], np.int64), it[0::2], it[1::2], T(b["cats"][0::2]), T(b["cats"][1::2]), T(b["ulab"]))
    dt = time.perf_counter() - t0
    val = B * steps / dt
    sample = f"{steps} steps of {B} BPR triples at full table size after {warm} warm-up (dense TF-1.x Adam sweep)"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warm, "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(cfg, B), "batch_triples": B, "optimizer": "adam (TF-1.x dense sweep)"},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "oracle restatement on torch-CPU, not TensorFlow (TF 1.x is not installable in this image)"}))


def workload_name(cfg, B):
    name = "cfg3" if cfg["U"] == CFG3["U"] else "cfg2"
    return (f"{name}: {cfg['U']} users x {cfg['I']} recipes x {cfg['L']} labels, D={cfg['D']}, "
            f"BPR B={B} triples/step, shuffled users, Zipf(1.05) positives")


def cpu_baseline_leg(cfg, B, budget_steps=3):
    """cpu_baseline of the default run: the same port, bounded to a few steps."""
    out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", str(budget_steps),
                          "--warmup", "1", "--batch", str(B)] + (["--small"] if cfg is SMALL else []),
                         capture_output=True, text=True, timeout=900,
                         env={k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")})
    for line in out.stdout.splitlines()[::-1]:
        if line.startswith("{"):
            return json.loads(line)["cpu_baseline"]
    return {"value": None, "unit": UNIT, "cores": len(os.sched_getaffinity(0)), "kind": "port",
            "sample": "failed: " + out.stderr[-300:]}


def cpu_catalog_leg(cfg, K=100, n_users=512):
    """CPU side of the catalog metric: the oracle's catalog_topk (float32 GEMM form on all host
    cores via BLAS + per-user lexsort) on a bounded sample of users over the full recipe table."""
    from oracle import evaluate_oracle
    from oracle.recommender_oracle import Hyper, OracleModel
    import synth_data as synth
    I, D = cfg["I"], cfg["D"]
    tb = synth.make_tables(n_users, I, 2, D, seed=3)
    ic = synth.make_item_categories(I)
    om = OracleModel(tb.P, tb.R, tb.Cat, tb.G, Hyper(), dtype=np.float32)
    t0 = time.perf_counter()
    evaluate_oracle.catalog_topk(om, np.arange(n_users), ic, K, dtype=np.float32)
    dt = time.perf_counter() - t0
    return {"value": n_users / dt, "unit": "users/s", "cores": len(os.sched_getaffinity(0)), "kind": "port",
            "sample": f"{n_users} users x {I} recipes, K={K}, float32 (oracle/evaluate_oracle.catalog_topk)"}


def cfg1_stream(n_batches, B=128):
    """BASELINE configs[0]: 10k users / 5k recipes / 95 labels / D=64 and the reference's own instance stream
    (get_train_instances, Train_recommender.py:74-96: user-contiguous, 1-2 users per 128-row batch)."""
    import synth_data as synth
    U, I, L, D = 10_000, 5_000, 95, 64
    tb = synth.make_tables(U, I, L, D, seed=synth.BASE_SEED + 1)
    ic = synth.make_item_categories(I); ul = synth.make_user_labels(U, L)
    train, _, tneg = synth.make_reference_dataset(max(8, n_batches * B // 50 + 8), I, seed=11)
    d2c, u2l = synth.reference_side_maps(ic, ul)
    u_idx, i_idx, labels, cats, sign, _ = synth.get_train_instances(train, tneg, d2c, u2l, seed=3)
    users = (np.asarray(u_idx).astype(np.int64) * 25 + 3) % U
    n = (len(users) // B) * B
    assert n >= n_batches * B, (n, n_batches)
    return tb, dict(users=users[:n].astype(np.int32), items=np.asarray(i_idx, np.int32)[:n],
                    labels=np.asarray(labels, np.float32)[:n], cats=np.asarray(cats, np.float32).reshape(-1, 4)[:n],
                    ws=np.asarray(sign, np.float32).reshape(-1)[:n], ulab=ul[users[:n]].astype(np.float32))


def cfg1_cpu_leg(steps=200, B=128):
    """The CPU arm at cfg1, exactly the reference's shape (pointwise, B=128, dense TF-1.x Adam sweep per step)."""
    import torch
    from oracle.cpu_port import CpuPort
    from oracle.recommender_oracle import Hyper
    cores = len(os.sched_getaffinity(0))
    tb, f = cfg1_stream(steps + 5, B)
    port = CpuPort(tb.P, tb.R, tb.Cat, tb.G, Hyper(learner="adam", lr=0.001), threads=cores)
    T = lambda k, dt=None: torch.as_tensor(f[k] if dt is None else f[k].astype(dt))
    tu, ti, ty, tc, tw, tl = T("users", np.int64), T("items", np.int64), T("labels"), T("cats"), T("ws"), T("ulab")
    t0 = None
    for k in range(steps + 5):
        if k == 5:
            t0 = time.perf_counter()
        sl = slice(k * B, (k + 1) * B)
        port.train_step(tu[sl], ti[sl], ty[sl], tc[sl], tw[sl], tl[sl])
    dt = time.perf_counter() - t0
    return {"value": B * steps / dt, "unit": "instances/s", "cores": cores, "kind": "port", "ms_per_step": 1e3 * dt / steps,
            "sample": f"{steps} pointwise steps of {B} rows of the reference stream at cfg1 (10k users, 5k recipes, D=64) after 5 warm-up"}


def cfg1_gpu_leg(dev, steps=200, B=128):
    """The CUDA path at cfg1 through the host entry point the drop-in Session uses: reference-format feed in pinned
    host memory, loss read on the host every step (what Train_recommender.py:195-200 does)."""
    import torch
    from foodrec_b200 import Engine, Hyper, _lib as L
    tb, f = cfg1_stream(steps + 5, B)
    eng = Engine(Hyper(learner="adam", lr=0.001), tb.P, tb.R, tb.Cat, tb.G, device=dev, max_rows=B, max_label_entries=B * 95)
    pin = {k: torch.as_tensor(np.ascontiguousarray(v)).pin_memory() for k, v in f.items()}
    launches0 = eng.lib.fr_launch_count()
    t0 = None
    for k in range(steps + 5):
        if k == 5:
            torch.cuda.synchronize(); t0 = time.perf_counter(); launches0 = eng.lib.fr_launch_count()
        sl = slice(k * B, (k + 1) * B)
        out = eng.train_step_host(L.FR_POINTWISE, B, pin["users"][sl], pin["items"][sl], pin["cats"][sl], pin["labels"][sl],
                                  pin["ws"][sl], pin["ulab"][sl])
        torch.cuda.current_stream().synchronize()
        loss = float(out[L.FR_OUT_LOSS])
    dt = time.perf_counter() - t0
    n_launch = eng.lib.fr_launch_count() - launches0
    eng.close()
    return {"value": B * steps / dt, "unit": "instances/s", "ms_per_step": 1e3 * dt / steps, "last_loss": loss,
            "launches_per_step": n_launch / steps,
            "note": "end to end (host feed in, loss out, synchronised every step); a 128-row step is launch-bound on a GPU"}


# ----------------------------------------------------------------------------- GPU arm, N > 1
def table_bytes(learner, bf16):
    """bytes per table ELEMENT: (a row read for scoring, the optimizer's read + write of the variable and its fp32 slots)"""
    slots = {"adam": 2, "adagrad": 1, "rmsprop": 2, "sgd": 0}[learner.lower()]
    vb = 2 if bf16 else 4
    return vb, 2 * vb + 8 * slots


def cfg5_leg(args, cfg, B, dev, steps, n_neg=8):
    """BASELINE configs[4] on ONE GPU: 1:8 sampled negatives (fr_sample_bpr_batch, Philox, drawn on the device inside the
    timed region), Adagrad, Personal_Memory / Recipe_Embedding stored in bf16 (fp32 arithmetic, RNE on store, fp32
    accumulators), the health term blended into sampled top-K at inference.  The same leg on fp32 tables runs beside it."""
    import torch
    from foodrec_b200 import Engine, Hyper, _lib as L
    import synth_data as synth
    U, I, Lb, D = cfg["U"], cfg["I"], cfg["L"], cfg["D"]
    item_cats = synth.make_item_categories(I)
    lab = synth.make_user_label_csr(U, Lb)
    n_pos = B // n_neg
    NB = 8
    pins = []
    for k in range(NB):
        rng = np.random.default_rng(5000 + k)
        pins.append((torch.as_tensor(rng.integers(0, U, n_pos).astype(np.int32)).pin_memory(),
                     torch.as_tensor(synth.zipf_items(rng, I, n_pos).astype(np.int32)).pin_memory()))
    devb = [(u.to(dev), p_.to(dev)) for u, p_ in pins]
    peak, peak_src = peaks()
    out = {}
    for td in ("float32", "bf16"):
        g = torch.Generator(device=dev); g.manual_seed(5)
        cast = (lambda x: x.to(torch.bfloat16)) if td == "bf16" else (lambda x: x)
        P = cast(torch.randn((U, 5, D), device=dev, generator=g) * 0.1); R = cast(torch.randn((I, D), device=dev, generator=g) * 0.1)
        Cat = torch.randn((4, D), device=dev, generator=g) * 0.1; G = torch.randn((Lb, 5, D), device=dev, generator=g) * 0.1
        eng = Engine(Hyper(learner="adagrad", lr=0.01), P, R, Cat, G, device=dev, max_rows=2 * B, item_cats=item_cats,
                     user_label_csr=lab, adopt=True, table_dtype=td)
        del P, R

        def step(k):
            u, p_ = devb[k % NB]
            eng.train_step_sampled(u, p_, n_neg, seed=20260105, sample_offset=k * n_pos)
        for k in range(10 + max(args.warmup, 3)):
            step(k)
        v = eng.read_scalars()
        uu, ui = float(v[L.FR_OUT_UNIQ_USERS]), float(v[L.FR_OUT_UNIQ_ITEMS])
        l0 = eng.lib.fr_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); e0.record()
        for k in range(steps):
            step(k)
        e1.record(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        launches = eng.lib.fr_launch_count() - l0
        eng.timing_enable(True)
        for k in range(steps):
            step(k)
        torch.cuda.synchronize()
        ph, _ = eng.timing_read()
        eng.timing_enable(False)
        rb, ub = table_bytes("adagrad", td == "bf16")
        alg = {"fwd": B * (7 * D * rb + 16), "user_chunk": uu * 5 * D * ub, "item_chunk": ui * D * ub}
        kern = {k: {"ms": ph[k], "alg_bytes": alg[k], "gbs": alg[k] / (ph[k] * 1e-3) / 1e9 if ph[k] > 0 else None} for k in alg}
        # the 8 triples of a positive share their user row and positive recipe row: the bytes that MUST come from HBM are
        # those of the distinct rows (the SURVEY 8(d) per-triple figure above counts every row of every triple)
        kern["fwd"]["distinct_row_bytes"] = uu * 5 * D * rb + ui * D * rb + B * 16
        step_bytes = alg["fwd"] + alg["user_chunk"] + alg["item_chunk"] + 4 * Lb * 5 * D
        dom = max(alg, key=lambda k: ph[k])
        # e2e: the (user, positive) pairs from pinned host memory, sampled + expanded on the device, loss read every step
        ub_, pb_ = torch.empty(n_pos, dtype=torch.int32, device=dev), torch.empty(n_pos, dtype=torch.int32, device=dev)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for k in range(steps):
            hu, hp = pins[k % NB]
            ub_.copy_(hu, non_blocking=True); pb_.copy_(hp, non_blocking=True)
            eng.train_step_sampled(ub_, pb_, n_neg, seed=20260105, sample_offset=k * n_pos)
            loss = float(eng.read_scalars()[L.FR_OUT_LOSS])
        dt = time.perf_counter() - t0
        # sampled top-K (51 candidates, K=10) with the health term blended in (fr_set_health_blend)
        NU = min(U, 1 << 20)
        rng = np.random.default_rng(5)
        eu = torch.as_tensor(rng.permutation(U)[:NU].astype(np.int32)).to(dev)
        cand = torch.as_tensor(rng.integers(0, I, (NU, 51)).astype(np.int32)).to(dev)
        nc = torch.full((NU,), 51, dtype=torch.int32, device=dev)
        eng.eval_sampled_topk(eu, cand, nc, 10); torch.cuda.synchronize()
        e0.record(); eng.eval_sampled_topk(eu, cand, nc, 10); e1.record(); torch.cuda.synchronize()
        ems_plain = e0.elapsed_time(e1)
        eng.set_health_blend(True)
        eng.eval_sampled_topk(eu, cand, nc, 10); torch.cuda.synchronize()
        e0.record(); eng.eval_sampled_topk(eu, cand, nc, 10); e1.record(); torch.cuda.synchronize()
        ems = e0.elapsed_time(e1)
        ealg = NU * (5 * D * rb + 51 * D * rb + 51 * 12)
        out[td] = {
            "metric": METRIC, "value": B / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "gpu_launches": int(launches),
            "phases_ms": {k: x for k, x in ph.items() if x > 0}, "kernels": kern,
            "roofline": {"bound": "hbm", "kernel": {"fwd": "fwd_train_kernel", "user_chunk": "seg_chunk_kernel<UserPol>",
                                                    "item_chunk": "seg_chunk_kernel<ItemPol>"}[dom],
                         "achieved": kern[dom]["gbs"], "peak": peak, "unit": "GB/s", "frac": kern[dom]["gbs"] / peak,
                         "peak_source": peak_src, "alg_bytes_per_launch": alg[dom], "ms_per_launch": ph[dom], "traffic": None},
            "roofline_step": {"bound": "hbm", "alg_bytes_per_step": step_bytes, "achieved": step_bytes / (ms * 1e-3) / 1e9,
                              "peak": peak, "unit": "GB/s", "frac": step_bytes / (ms * 1e-3) / 1e9 / peak},
            "e2e": {"value": B * steps / dt, "unit": UNIT, "h2d_bytes_per_step": 8 * n_pos, "d2h_bytes_per_step": 4 * L.FR_OUT_COUNT,
                    "feed": "(user, positive) pairs from pinned host memory; negatives drawn and the batch expanded on the device; "
                            "loss read every step", "last_loss": loss},
            "topk_health": {"metric": "sampled_topk_users_per_sec", "value": NU / (ems * 1e-3), "unit": "users/s", "ms": ems,
                            "users": NU, "candidates": 51, "K": 10,
                            "roofline": {"bound": "hbm", "achieved": ealg / (ems * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                                         "frac": ealg / (ems * 1e-3) / 1e9 / peak},
                            "note": "the health term adds the user's General_Memory rows (<= 3 labels x 5 x D floats, L2-resident) "
                                    "to every user's reads; they are not in the algorithmic byte count"},
            "topk": {"metric": "sampled_topk_users_per_sec", "value": NU / (ems_plain * 1e-3), "unit": "users/s", "ms": ems_plain,
                     "users": NU, "candidates": 51, "K": 10, "health_term": False,
                     "roofline": {"bound": "hbm", "achieved": ealg / (ems_plain * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                                  "frac": ealg / (ems_plain * 1e-3) / 1e9 / peak}},
            "uniq_users_per_step": uu, "uniq_items_per_step": ui,
        }
        eng.close(); del eng
        torch.cuda.empty_cache()
    res = out["bf16"]
    res["workload"] = (f"cfg5 (BASELINE configs[4]) on one GPU: {U} users x {I} recipes x {Lb} labels, D={D}; {n_pos} positives x "
                       f"{n_neg} sampled negatives = {B} BPR triples per step; Adagrad; bf16 Personal_Memory / Recipe_Embedding "
                       "(fp32 arithmetic and accumulators, round-to-nearest-even on store); health term at inference")
    res["dtype"] = "f32 arithmetic, bf16 table storage"
    f = out["float32"]
    res["same_leg_fp32_tables"] = {"value": f["value"], "ms_per_step": f["ms_per_step"], "phases_ms": f["phases_ms"],
                                   "roofline_step_frac": f["roofline_step"]["frac"], "topk_health_ms": f["topk_health"]["ms"],
                                   "topk_ms": f["topk"]["ms"],
                                   "e2e": f["e2e"]["value"]}
    res["speedup_vs_fp32_tables"] = res["value"] / f["value"]
    return res


def shard_self_check(rank, world, dev, p2p):
    """Correctness of the N-rank step IN the bench run (the 2-GPU pytest cannot run on a 1-GPU lease): a small problem is
    trained for a few steps through the same DistRunner (same collectives, same peer-store path) while rank 0 trains
    an unsharded Engine on the same global batches; every rank's rows are gathered and compared element-wise."""
    import torch
    import torch.distributed as dist
    from foodrec_b200 import Engine, Hyper
    from foodrec_b200 import sharded as sh
    import synth_data as synth
    U, I, Lb, D, B = 8192 * world + 3, 4099, 95, 128, 2048 * world
    tb = synth.make_tables(U, I, Lb, D, seed=5)
    ic = synth.make_item_categories(I, seed=6)
    off, idx = synth.make_user_label_csr(U, Lb, seed=7)
    hy = Hyper(learner="adam", lr=0.01)
    eng = sh.ShardedEngine(hy, sh.shard_rows(tb.P, rank, world), sh.shard_rows(tb.R, rank, world), tb.Cat, tb.G, rank, world,
                           device=dev, max_rows=2 * B, item_cats_global=ic,
                           user_label_csr_local=sh.shard_label_csr(off, idx, rank, world, U))
    run = sh.DistRunner(eng)
    if p2p:
        run.enable_p2p()
    single = Engine(hy, tb.P, tb.R, tb.Cat, tb.G, device=dev, max_rows=2 * B, item_cats=ic, user_label_csr=(off, idx)) if rank == 0 else None
    worst_loss = 0.0
    for s in range(4):
        rng = np.random.default_rng(40 + s)                     # the same global batch on every rank
        users = rng.integers(0, U, B).astype(np.int32)
        if s == 2:
            users[: B // 2] = users[0]                          # a heavy user: long runs, one rank far busier than the others
        pos = synth.zipf_items(rng, I, B)
        neg = rng.integers(0, I, B).astype(np.int32); neg[neg == pos] = (neg[neg == pos] + 1) % I
        ix = sh.route_batch(users, world)[rank]
        eng.set_batch(users[ix] // world, pos[ix], neg_items=neg[ix], global_batch=B)
        out = run.step().cpu().numpy()
        assert out[9] == 0, "capacity / id flag raised in the self-check"
        if single is not None:
            single.train_step(users, pos, neg_items=neg)
            v = single.read_scalars()
            worst_loss = max(worst_loss, abs(out[0] - v[0]) / abs(v[0]))
    eng.e.flush()
    Pl, Rl = eng.e.P.contiguous(), eng.e.R.contiguous()
    Ps = [torch.empty_like(Pl) for _ in range(world)]; Rs = [torch.empty_like(Rl) for _ in range(world)]
    dist.all_gather(Ps, Pl); dist.all_gather(Rs, Rl)
    res = None
    if rank == 0:
        t = single.tables()
        def rel(x, ref):
            ref = ref.astype(np.float64)
            return float(np.max(np.abs(x.astype(np.float64) - ref) / np.maximum(np.abs(ref), np.sqrt(np.mean(ref ** 2)))))
        errs = {"P": rel(sh.unshard_rows([x.cpu().numpy() for x in Ps], U), t["P"]),
                "R": rel(sh.unshard_rows([x.cpu().numpy() for x in Rs], I), t["R"]),
                "Cat": rel(eng.e.Cat.cpu().numpy(), t["Cat"]), "G": rel(eng.e.G.cpu().numpy(), t["G"])}
        # Adam: summation order differs between the sharded and the unsharded step (recipe gradients are pre-reduced per
        # rank): 1e-4 on P / R / Cat as in tests/test_gpu_sharded.py, 1e-5 on G and the loss
        ok = worst_loss <= 1e-5 and errs["G"] <= 1e-5 and max(errs["P"], errs["R"], errs["Cat"]) <= 1e-4
        res = {"ok": bool(ok), "steps": 4, "users": U, "recipes": I, "global_batch": B, "loss_rel_err": worst_loss,
               "table_rel_err": errs, "compared": "every row of every rank, all-gathered, against an unsharded engine on rank 0"}
        single.close()
    eng.e.close()
    del eng, run
    torch.cuda.empty_cache()
    flag = torch.tensor([1.0 if (res is None or res["ok"]) else 0.0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if float(flag.item()) != 1.0:
        if rank == 0:
            print(json.dumps({"self_check": res}), file=sys.stderr)
        raise SystemExit("sharded self-check FAILED: the N-rank step does not reproduce the unsharded engine")
    return res


def sharded_train_leg(args, cfg_local, B, rank, world, dev, p2p, steps, preroll, warmup, label, single_pass=None,
                      learner=None, table_dtype="float32", n_neg=0, extras=True):
    """One weak-scaling training measurement: every rank holds `cfg_local` rows (its shard), B triples per rank per step.
    n_neg > 0: B/n_neg (user, positive) pairs per rank, negatives drawn on the device over the global catalog
    (fr_sample_bpr_batch) inside the timed region.  extras=False: no e2e / un-routed legs."""
    import torch
    import torch.distributed as dist
    from foodrec_b200 import Hyper, _lib as L
    from foodrec_b200.sharded import DistRunner, ShardedEngine
    import synth_data as synth
    Ul, Il, Lb, D = cfg_local["U"], cfg_local["I"], cfg_local["L"], cfg_local["D"]
    I = Il * world
    learner = learner or args.learner
    bf16 = table_dtype == "bf16"
    g = torch.Generator(device=dev); g.manual_seed(1 + rank)
    P = torch.empty((Ul, 5, D), device=dev).normal_(0, 0.1, generator=g); R = torch.empty((Il, D), device=dev).normal_(0, 0.1, generator=g)
    if bf16:
        P, R = P.to(torch.bfloat16), R.to(torch.bfloat16)
    g2 = torch.Generator(device=dev); g2.manual_seed(99)          # replicated tables: same on every rank
    Cat = torch.randn((4, D), device=dev, generator=g2) * 0.1; G = torch.randn((Lb, 5, D), device=dev, generator=g2) * 0.1
    item_cats = synth.make_item_categories(I)
    lab = synth.make_user_label_csr(Ul, Lb, seed=synth.BASE_SEED + 200 + rank)
    eng = ShardedEngine(Hyper(learner=learner, lr=0.001), P, R, Cat, G, rank, world, device=dev, max_rows=2 * B + 16384,
                        adam_mode=args.adam_mode, item_cats_global=item_cats, user_label_csr_local=lab, adopt=True,
                        single_pass=single_pass, table_dtype=table_dtype)
    # (+16384 rows: an un-routed batch lands B +- a few hundred groups per rank)
    del P, R
    run = DistRunner(eng)
    if p2p:
        run.enable_p2p()
    NB = 8
    pin, devb = [], []
    for k in range(NB):
        rng = np.random.default_rng(1000 + 100 * rank + k)
        users = rng.integers(0, Ul, B).astype(np.int32)            # LOCAL user rows: this rank owns them
        pos = synth.zipf_items(rng, I, B)
        neg = rng.integers(0, I, B).astype(np.int32); neg[neg == pos] = (neg[neg == pos] + 1) % I
        items = np.stack([pos, neg], 1).reshape(-1).copy()
        if n_neg:
            users, items = users[:B // n_neg].copy(), pos[:B // n_neg].astype(np.int32)
        pin.append((torch.as_tensor(users).pin_memory(), torch.as_tensor(items).pin_memory()))
        devb.append((pin[-1][0].to(dev), pin[-1][1].to(dev)))

    def setb(k):
        u, it = devb[k % NB]
        if n_neg:
            eng.set_batch_sampled(u, it, n_neg, seed=20260105, sample_offset=(k * world + rank) * (B // n_neg), global_batch=world * B)
        else:
            eng.set_batch_dev(L.FR_BPR, B, u, it, global_batch=world * B)

    def step(k, **kw):
        # the NEXT step's fr_shard_plan + id all-to-all ride on a side stream under this step's update / apply
        if not eng.planned():
            setb(k)
        return run.step(next_batch=None if args.no_plan_ahead else (lambda: setb(k + 1)), **kw)

    for k in range(preroll + warmup):
        step(k)
    v = eng.e.read_scalars()
    launches0 = eng.e.lib.fr_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    dist.barrier(); torch.cuda.synchronize()
    t_begin = time.time()
    ev0.record()
    for k in range(steps):
        step(k)
    ev1.record()
    dist.barrier(); torch.cuda.synchronize()
    t_end = time.time()
    launches = eng.e.lib.fr_launch_count() - launches0
    t = torch.tensor([ev0.elapsed_time(ev1)], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); ms = float(t.item())
    # per-kernel events inside the library (rank 0's numbers) and per-phase events around every fr_shard_* call / collective
    n_ph = min(steps, 10)
    eng.e.timing_enable(True)
    for k in range(n_ph):
        step(k)
    torch.cuda.synchronize()
    sphases, _ = eng.e.timing_read()
    eng.e.timing_enable(False)
    shard_ms = {}
    for k in range(n_ph):
        evs = []
        step(k, phase_events=evs)
        torch.cuda.synchronize()
        for (name, e0), (_, e1) in zip(evs[:-1], evs[1:]):
            shard_ms[name] = shard_ms.get(name, 0.0) + e0.elapsed_time(e1) / n_ph
    v = eng.e.read_scalars()
    peak, peak_src = peaks()
    rb, upd = table_bytes(learner, bf16)
    adam_k = upd / 4                     # (fp32: 6 for Adam = var + m + v read and written; kept as a factor of 4-byte words)
    uu, ui = float(v[L.FR_OUT_UNIQ_USERS]), float(v[L.FR_OUT_UNIQ_ITEMS])
    fused = bool(eng.e.single_pass)
    # dominant kernel on rank 0: the single-pass kernel lives in the `forward` phase, the two-pass user pass in `update`
    if fused:
        kms = shard_ms.get("forward", 0.0)
        kalg = uu * adam_k * 20 * D + B * (2 * 4 * D + 16) + B * 2 * 4 * D
        kname, kscope = "user_fused_kernel (+ label scatter: the `forward` phase)", "phase time, per GPU (rank 0)"
    else:
        kms = sphases.get("user_chunk", 0.0)
        kalg = uu * adam_k * 20 * D
        kname, kscope = "seg_chunk_kernel<UserPol>", "per GPU (rank 0)"
        if sphases.get("fwd", 0.0) > kms:           # (1:8 sampled negatives: few distinct users, the forward dominates)
            kms, kalg, kname = sphases["fwd"], B * (7 * D * rb + 16), "fwd_train_kernel"
    sroof = None
    if kms > 0:
        sroof = {"bound": "hbm", "kernel": kname, "achieved": kalg / (kms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                 "frac": kalg / (kms * 1e-3) / 1e9 / peak, "peak_source": peak_src, "alg_bytes_per_launch": kalg,
                 "ms_per_launch": kms, "scope": kscope, "traffic": None}
    step_bytes = B * (7 * D * rb + 16) + uu * adam_k * 20 * D + ui * adam_k * 4 * D + 4 * Lb * 5 * D
    if not extras:
        res = {
            "label": label, "value": world * B * steps / (ms / 1e3), "unit": UNIT, "ms_per_step": ms / steps, "steps": steps,
            "launches": int(launches), "window": (t_begin, t_end), "p2p": p2p, "cap": eng.cap, "optimizer": learner,
            "table_dtype": table_dtype, "sampled_negatives_per_positive": n_neg,
            "local_rows": {"users": Ul, "recipes": Il}, "global_rows": {"users": Ul * world, "recipes": I},
            "roofline": sroof, "shard_phases_ms": shard_ms, "update_phase_kernels_ms": {k: sphases[k] for k in sphases if sphases[k] > 0},
            "roofline_step": {"bound": "hbm", "alg_bytes_per_step_per_gpu": step_bytes, "achieved": step_bytes / (ms / steps * 1e-3) / 1e9,
                              "peak": peak, "unit": "GB/s", "frac": step_bytes / (ms / steps * 1e-3) / 1e9 / peak, "scope": "per GPU"},
            "uniq_users_per_step": uu, "uniq_items_per_step": ui, "overflow_flag": float(v[L.FR_OUT_OVERFLOW])}
        return res, eng, run
    # e2e, both feeds: ids only (side tables resident) and the reference's dense feed (categories + user_one_hot_label)
    ubuf = torch.empty(B, dtype=torch.int32, device=dev); ibuf = torch.empty(2 * B, dtype=torch.int32, device=dev)

    def e2e(dense):
        hc = hl = dc = dl = None
        if dense:
            hc = [torch.as_tensor(item_cats[pin[k][1].numpy()]).pin_memory() for k in range(NB)]
            hl = [torch.as_tensor(synth.csr_rows_dense(lab[0], lab[1], pin[k][0].numpy(), Lb)).pin_memory() for k in range(NB)]
            dc = torch.empty((2 * B, 4), dtype=torch.float32, device=dev); dl = torch.empty((B, Lb), dtype=torch.float32, device=dev)
        dist.barrier(); torch.cuda.synchronize()
        t0 = time.perf_counter()
        loss = 0.0
        for k in range(steps):
            hu, hi = pin[k % NB]
            ubuf.copy_(hu, non_blocking=True); ibuf.copy_(hi, non_blocking=True)
            if eng.planned():                                   # a plan left over from a pipelined leg: run it out
                run.step()
            if dense:
                dc.copy_(hc[k % NB], non_blocking=True); dl.copy_(hl[k % NB], non_blocking=True)
                eng.set_batch_raw(L.fr_batch(L.FR_BPR, B, ubuf.data_ptr(), ibuf.data_ptr(), dc.data_ptr(), None, None, dl.data_ptr()),
                                  [ubuf, ibuf, dc, dl], world * B)
            else:
                eng.set_batch_dev(L.FR_BPR, B, ubuf, ibuf, global_batch=world * B)
            out = run.step()
            loss = float(out[L.FR_OUT_LOSS])                      # D2H + sync
        dist.barrier(); torch.cuda.synchronize()
        tt = torch.tensor([time.perf_counter() - t0], device=dev); dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return world * B * steps / float(tt.item()), loss
    e2e_ids, loss_ids = e2e(False)
    e2e_dense, _ = e2e(True)
    # un-routed stream: every rank receives B triples of ARBITRARY users (global ids); fr_shard_route buckets them by
    # owner, one all-to-all moves them, fr_shard_unroute compacts -- then the same step.  Device-timed, max over ranks.
    gb = []
    for k in range(NB):
        rng = np.random.default_rng(7000 + 100 * rank + k)
        users = rng.integers(0, Ul * world, B).astype(np.int32)
        pos = synth.zipf_items(rng, I, B)
        neg = rng.integers(0, I, B).astype(np.int32); neg[neg == pos] = (neg[neg == pos] + 1) % I
        gb.append((torch.as_tensor(users).to(dev), torch.as_tensor(np.stack([pos, neg], 1).reshape(-1).copy()).to(dev)))

    def uset(k):
        u, it = gb[k % NB]
        run.set_batch_unrouted(L.FR_BPR, u, it, global_batch=world * B)

    def ustep(k):
        # routing of batch k+1 (bucket, all-to-all, compaction, the host read of its size) rides on the side stream
        # under step k, like the plan: the timed region contains every routing call
        if not eng.planned() and eng._pending is None:
            uset(k)
        return run.step(next_batch=None if args.no_plan_ahead else (lambda: uset(k + 1)))
    while eng.planned():                                    # a plan left over from the pipelined legs: run it out
        run.step()
    for k in range(3):
        ustep(k)
    u0, u1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    dist.barrier(); torch.cuda.synchronize()
    u0.record()
    for k in range(steps):
        ustep(k)
    u1.record()
    dist.barrier(); torch.cuda.synchronize()
    tt = torch.tensor([u0.elapsed_time(u1)], device=dev); dist.all_reduce(tt, op=dist.ReduceOp.MAX); ums = float(tt.item())
    while eng.planned():
        run.step()
    ra, rb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)       # routing alone, un-overlapped
    torch.cuda.synchronize(); ra.record()
    for k in range(5):
        uset(k)
    rb.record(); torch.cuda.synchronize()
    route_ms = ra.elapsed_time(rb) / 5
    eng._pending = None
    unrouted = {"value": world * B * steps / (ums / 1e3), "unit": UNIT, "ms_per_step": ums / steps, "route_ms_alone_rank0": route_ms,
                "exchange_bytes_per_gpu": int(eng._rsend.numel() * 4 * (world - 1) / world),
                "note": "samples arrive on a random rank: bucket by owner + ONE all-to-all + compaction (fr_shard_route / "
                        "fr_shard_unroute) inside the timed region, issued one step ahead on the side stream like the plan; "
                        "the routed size is read on the host every step"}
    res = {
        "label": label, "value": world * B * steps / (ms / 1e3), "ms_per_step": ms / steps, "steps": steps, "launches": int(launches),
        "window": (t_begin, t_end), "single_pass": fused, "p2p": p2p, "cap": eng.cap,
        "local_rows": {"users": Ul, "recipes": Il}, "global_rows": {"users": Ul * world, "recipes": I},
        "roofline": sroof, "shard_phases_ms": shard_ms, "update_phase_kernels_ms": {k: sphases[k] for k in sphases if sphases[k] > 0},
        "roofline_step": {"bound": "hbm", "alg_bytes_per_step_per_gpu": step_bytes, "achieved": step_bytes / (ms / steps * 1e-3) / 1e9,
                          "peak": peak, "unit": "GB/s", "frac": step_bytes / (ms / steps * 1e-3) / 1e9 / peak, "scope": "per GPU"},
        "e2e": {"value": e2e_dense, "unit": UNIT, "h2d_bytes_per_step": B * (12 + 2 * 16 + 4 * Lb), "d2h_bytes_per_step": 4 * L.FR_OUT_COUNT,
                "feed": "reference dense feed (user_input, item_input, categories, user_one_hot_label) from pinned host memory, "
                        "loss read every step -- the same feed as the N=1 e2e"},
        "e2e_compact": {"value": e2e_ids, "unit": UNIT, "h2d_bytes_per_step": 12 * B,
                        "feed": "ids only (user, pos, neg); side tables resident", "last_loss": loss_ids},
        "unrouted": unrouted, "uniq_users_per_step": uu, "uniq_items_per_step": ui, "overflow_flag": float(v[L.FR_OUT_OVERFLOW]),
    }
    return res, eng, run


def run_sharded(args, cfg, B):
    """N GPUs of one node, one process per GPU: tables row-sharded (P by user % N, R by recipe % N), B triples per GPU
    per step, every triple loaded on the rank that owns its user; recipe rows and their gradients cross NVLink (peer
    stores from inside the gather / gradient kernels, or staged all-to-alls), one packed all-reduce per step.
    WEAK SCALING AT CONSTANT PER-GPU WORK: every GPU holds a cfg2-sized Personal_Memory shard (1M users per GPU: the
    user table grows with N, the 200k-recipe catalog is sharded), so the unique user rows a GPU touches per step are
    those of the N=1 run (--fixed-tables: round-1 behaviour, the 1M users divided over the ranks).  value = N*B*K / max-over-ranks device time."""
    import torch
    import torch.distributed as dist
    from foodrec_b200 import Hyper
    from foodrec_b200.sharded import DistRunner, ShardedEngine, local_rows
    import synth_data as synth
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    clocks = ClockSampler(local); clocks.start()
    dist.init_process_group("nccl", device_id=dev)
    U, I, Lb, D = cfg["U"], cfg["I"], cfg["L"], cfg["D"]
    p2p = not args.no_p2p
    if p2p:
        try:
            import torch.distributed._symmetric_memory  # noqa: F401
        except Exception as ex:
            p2p = False
            if rank == 0:
                print(f"peer-memory exchange unavailable ({type(ex).__name__}: {ex}); using all-to-alls", file=sys.stderr)
    check = shard_self_check(rank, world, dev, p2p)
    if args.cfg3 or args.fixed_tables:
        cfg_local = dict(U=local_rows(U, world), I=local_rows(I, world), L=Lb, D=D)
        mode = "cfg3 (BASELINE configs[2])" if args.cfg3 else "fixed tables (cfg2 divided over the ranks)"
    else:
        cfg_local = dict(U=U, I=local_rows(I, world), L=Lb, D=D)
        mode = f"constant per-GPU work: {U} users PER GPU ({U * world} in all), the {I}-recipe catalog sharded over the ranks"
    main, eng, run = sharded_train_leg(args, cfg_local, B, rank, world, dev, p2p, args.steps, args.preroll, args.warmup, mode)
    clocks.t0, clocks.t1 = main.pop("window")
    clk = clocks.stop()
    Ul, Il = cfg_local["U"], cfg_local["I"]
    I_glob = Il * world
    # ---- item-sharded full-catalog top-100: n_q query users PER GPU (weak scaling), recipes sharded by id % N:
    # all-gather of the query rows, per-shard tcgen05 top-K, all-to-all of the lists, exact merge
    catalog = None
    if not args.no_catalog:
        n_q = min(18_944, Ul)
        eng.catalog_prepare()
        ul = torch.arange(n_q, dtype=torch.int32, device=dev)
        run.catalog_topk(ul, K=100)
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        dist.barrier(); torch.cuda.synchronize()
        c0.record(); cid, csc = run.catalog_topk(ul, K=100); c1.record()
        dist.barrier(); torch.cuda.synchronize()
        t = torch.tensor([c0.elapsed_time(c1)], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); cms = float(t.item())
        catalog = {"metric": "catalog_topk_users_per_sec", "value": world * n_q / (cms * 1e-3), "unit": "users/s",
                   "workload": f"{n_q} query users per GPU x {I_glob} recipes sharded by id % {world}, D={D}, K=100",
                   "ms": cms, "fallback_rows_rank0": eng.e.catalog_fallback_rows(), "train_steps_before": int(eng.e.step),
                   "exchange_bytes_per_gpu": {"all_gather_rows": (world - 1) * n_q * 5 * D * 4,
                                              "all_to_all_lists": (world - 1) * n_q * 100 * 12}}
    Cat, G = eng.e.Cat.clone(), eng.e.G.clone()
    eng.e.close(); del eng, run
    torch.cuda.empty_cache()
    if not args.no_catalog and not args.small and not args.cfg3:
        # cfg4 shape (BASELINE configs[3]): 10M recipes item-sharded over the N GPUs.  FULL query set: 1M users in all,
        # 1M / N per GPU in blocks of n_q (every GPU scores every gathered block against its recipe shard)
        I4, U4 = 10_000_000, 1_000_000
        Il4 = local_rows(I4, world)
        n_q = 18_944
        per_gpu = -(-U4 // world)
        blocks = -(-per_gpu // n_q)
        g4 = torch.Generator(device=dev); g4.manual_seed(40 + rank)
        e4 = ShardedEngine(Hyper(learner="sgd"), torch.randn((n_q * blocks, 5, D), device=dev, generator=g4) * 0.1,
                           torch.randn((Il4, D), device=dev, generator=g4) * 0.1, Cat, G, rank, world, device=dev,
                           max_rows=256, item_cats_global=synth.make_item_categories(I4), adopt=True)
        e4.e.I_global = I4
        e4.catalog_prepare()
        run4 = DistRunner(e4)
        ul = torch.arange(n_q, dtype=torch.int32, device=dev)
        run4.catalog_topk(ul, K=100)
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        dist.barrier(); torch.cuda.synchronize()
        c0.record()
        fb = 0
        for bk in range(blocks):
            run4.catalog_topk(ul + bk * n_q, K=100)
        c1.record()
        dist.barrier(); torch.cuda.synchronize()
        t = torch.tensor([c0.elapsed_time(c1)], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); cms4 = float(t.item())
        n_users4 = world * n_q * blocks
        catalog = [catalog, {
            "metric": "catalog_topk_users_per_sec", "value": n_users4 / (cms4 * 1e-3), "unit": "users/s",
            "workload": f"cfg4 IN FULL: {n_users4} query users ({n_q * blocks} per GPU in {blocks} blocks of {n_q}) x {I4} recipes "
                        f"sharded by id % {world}, D={D}, K=100; all-gather of query rows, per-shard top-K, all-to-all of the lists, merge",
            "ms": cms4, "fallback_rows_rank0_last_block": e4.e.catalog_fallback_rows(),
            "dense_equivalent_tflops_per_gpu": 2.0 * n_users4 * Il4 * 5 * D / (cms4 * 1e-3) / 1e12}]
        e4.e.close(); del e4, run4
        torch.cuda.empty_cache()
    # ---- BASELINE configs[4]: 1:8 sampled negatives, Adagrad, bf16 tables, row-sharded like the main leg (and the same
    # leg on fp32 tables beside it)
    cfg5_line = None
    if not args.small and not args.cfg3 and not args.no_cfg5:
        c5 = {}
        for td in ("float32", "bf16"):
            c5[td], e5, r5 = sharded_train_leg(args, cfg_local, B, rank, world, dev, p2p, args.steps, 10, 3,
                                               "cfg5 (BASELINE configs[4]): 1:8 sampled negatives, Adagrad, " + td + " tables; " + mode,
                                               single_pass=False, learner="adagrad", table_dtype=td, n_neg=8, extras=False)
            c5[td].pop("window")
            e5.e.close(); del e5, r5
            torch.cuda.empty_cache()
        cfg5_line = c5["bf16"]
        cfg5_line["same_leg_fp32_tables"] = {k: c5["float32"][k] for k in ("value", "ms_per_step", "shard_phases_ms", "update_phase_kernels_ms")}
        cfg5_line["speedup_vs_fp32_tables"] = c5["bf16"]["value"] / c5["float32"]["value"]
    # ---- BASELINE configs[2] at N = 8: 100M users / 10M recipes row-sharded (12.5M users = 96 GB of P + Adam slots per
    # GPU: no room for the single-pass shadow copy -> two-pass step), fewer steps (the tables take a while to fill)
    cfg3_line = None
    if world == 8 and not args.small and not args.cfg3 and not args.no_cfg3:
        c3 = dict(U=local_rows(CFG3["U"], world), I=local_rows(CFG3["I"], world), L=Lb, D=D)
        cfg3_line, e3, r3 = sharded_train_leg(args, c3, B, rank, world, dev, p2p, min(args.steps, 20), 12, 3,
                                              "cfg3 (BASELINE configs[2]): 100M users / 10M recipes over 8 GPUs", single_pass=False)
        cfg3_line.pop("window")
        e3.e.close(); del e3, r3
        torch.cuda.empty_cache()
    # ---- BASELINE configs[4] at SURVEY 8(d)'s sizes (cfg3's: 100M users / 10M recipes), N = 8: 1:8 sampled negatives,
    # Adagrad, bf16 tables -- 16 GB of Personal_Memory + 32 GB of fp32 accumulators per GPU
    # (FOODREC_CFG5_BIG_USERS / _RECIPES: totals for a dry run of this leg at another N)
    cfg5_big = None
    big_u = int(os.environ.get("FOODREC_CFG5_BIG_USERS", CFG3["U"] if world == 8 else 0))
    big_i = int(os.environ.get("FOODREC_CFG5_BIG_RECIPES", CFG3["I"]))
    if big_u and not args.small and not args.cfg3 and not args.no_cfg3 and not args.no_cfg5:
        try:
            c5b = dict(U=local_rows(big_u, world), I=local_rows(big_i, world), L=Lb, D=D)
            cfg5_big, e5, r5 = sharded_train_leg(args, c5b, B, rank, world, dev, p2p, min(args.steps, 20), 8, 3,
                                                 f"cfg5 at cfg3's sizes: {big_u} users / {big_i} recipes over {world} GPUs, 1:8 sampled "
                                                 "negatives, Adagrad, bf16 tables", single_pass=False, learner="adagrad",
                                                 table_dtype="bf16", n_neg=8, extras=False)
            cfg5_big.pop("window")
            e5.e.close(); del e5, r5
            torch.cuda.empty_cache()
        except Exception as ex:          # (every rank runs the same leg on the same shapes: a failure is one on all ranks)
            cfg5_big = {"error": f"{type(ex).__name__}: {ex}"[:300]}
    if rank == 0:
        line = {
            "metric": METRIC, "value": main["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "catalog_topk": catalog,
            "config": {"workload": workload_name(dict(cfg, U=Ul * world, I=I_glob), B) + f" PER GPU (global batch {world * B}); " + mode,
                       "batch_triples": B,
                       "optimizer": (f"adam (TF-1.x semantics, {args.adam_mode})" if args.learner.lower() == "adam" else args.learner),
                       "l2": "per-step working set >> 126 MB L2; 8 distinct batches cycled", "preroll_steps": args.preroll,
                       "parallelism": f"row-sharded x{world}: P by user%N (samples loaded at the user owner), R by recipe%N; " + (
                           f"id all-to-all + recipe rows / gradient rows stored into peer memory over NVLink by the gather / "
                           f"gradient kernels (cap {main['cap']}/pair, 2 barriers) + 1 packed all-reduce per step" if p2p else
                           f"3 all-to-alls (ids, rows, grad rows, cap {main['cap']}/pair) + 1 packed all-reduce per step")},
            "clocks": clk, "gpu_launches": main["launches"], "roofline": main["roofline"], "roofline_step": main["roofline_step"],
            "single_pass": main["single_pass"], "shard_phases_ms": main["shard_phases_ms"],
            "update_phase_kernels_ms": main["update_phase_kernels_ms"], "self_check": check,
            "e2e": main["e2e"], "e2e_compact": main["e2e_compact"], "unrouted": main["unrouted"],
            "uniq_users_per_step": main["uniq_users_per_step"], "uniq_items_per_step": main["uniq_items_per_step"],
            "overflow_flag": main["overflow_flag"], "cfg3": cfg3_line, "cfg5": cfg5_line, "cfg5_cfg3_sizes": cfg5_big}
        print(json.dumps(line, default=float))
    dist.destroy_process_group()


# ----------------------------------------------------------------------------- GPU arm
DUMP_ROWS = {"P": 8192, "R": 16384}      # sampled rows of the two large tables: 21 MB + 8 MB at D=128


def dump_outputs(out_dir, eng):
    """--dump-outputs: what the last timed step hands its caller, as float32 DIR/<name>.npy -- the step's scalar
    vector (FR_OUT_*: loss, norm, clip scale, ...) and the tables it updated: Category_Embedding and General_Memory
    whole, Personal_Memory and Recipe_Embedding as a fixed seeded sample of rows (the full tables are GBs).  The
    sample depends only on the table sizes, so two builds run with the same arguments compare row for row."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    out = {"scalars": eng.read_scalars()}
    eng.flush()                          # lazy Adam: every row brought to the current step, as Engine.tables() does
    for k, n in DUMP_ROWS.items():
        t = getattr(eng, k)
        rows = np.sort(np.random.default_rng(2026).choice(t.shape[0], min(n, t.shape[0]), replace=False))
        out[k + "_sample"] = t[torch.as_tensor(rows, device=t.device)].float().cpu().numpy()
    out["Cat"], out["G"] = eng.Cat.float().cpu().numpy(), eng.G.float().cpu().numpy()
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, np.float32))


def run_ours(args, cfg, B):
    import torch
    import torch.distributed as dist
    from foodrec_b200 import Engine, Hyper, _lib as L
    import synth_data as synth      # input generator only; nothing under oracle/ runs in this arm
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    full_affinity = os.sched_getaffinity(0)
    numa = bind_to_gpu_numa_node(local)
    clocks = ClockSampler(local); clocks.start()      # early: nvidia-smi takes ~1 s to emit its first sample
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    U, I, Lb, D = cfg["U"], cfg["I"], cfg["L"], cfg["D"]
    g = torch.Generator(device=dev); g.manual_seed(1 + rank)
    P = torch.randn((U, 5, D), device=dev, generator=g) * 0.1; R = torch.randn((I, D), device=dev, generator=g) * 0.1
    Cat = torch.randn((4, D), device=dev, generator=g) * 0.1; G = torch.randn((Lb, 5, D), device=dev, generator=g) * 0.1
    item_cats = synth.make_item_categories(I)
    lab = synth.make_user_label_csr(U, Lb)
    eng = Engine(Hyper(learner=args.learner, lr=0.001), P, R, Cat, G, device=dev, max_rows=2 * B,
                 adam_mode=args.adam_mode, item_cats=item_cats, user_label_csr=lab)
    # (label-entry capacity defaults to rows x max labels per user = 2B x 3: sized to the data)
    del P
    NB = 8
    host = make_batches(cfg, B, NB, 1000 + 100 * rank, item_cats, lab, dense=True)
    dev_b = [(torch.as_tensor(b["users"]).to(dev), torch.as_tensor(b["items"]).to(dev)) for b in host]

    def step(k):
        u, it = dev_b[k % NB]
        eng._step_dev(L.FR_BPR, B, u, it, None, None, None, None)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # steady state for lazy Adam: most rows have live moments before anything is timed
    preroll = args.preroll
    for k in range(preroll):
        step(k)
    for k in range(args.warmup):
        step(preroll + k)
    v = eng.read_scalars()
    uniq_users, uniq_items = float(v[L.FR_OUT_UNIQ_USERS]), float(v[L.FR_OUT_UNIQ_ITEMS])
    # ---- timed region: device timing, inputs resident in HBM
    launches0 = eng.lib.fr_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    clocks.mark_begin()
    ev0.record()
    for k in range(args.steps):
        step(k)
    ev1.record()
    barrier()
    clocks.mark_end()
    launches = eng.lib.fr_launch_count() - launches0
    ms = ev0.elapsed_time(ev1)
    if world > 1:
        t = torch.tensor([ms], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); ms = float(t.item())
    clk = clocks.stop()
    value = world * B * args.steps / (ms / 1e3)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, eng)     # before the legs below train the same tables further

    # ---- per-kernel timing (CUDA events inside fr_train_step, on its stream), same steps again
    eng.timing_enable(True)
    for k in range(args.steps):
        step(k)
    torch.cuda.synchronize()
    phases, nst = eng.timing_read()
    eng.timing_enable(False)
    peak, peak_src = peaks()
    adam_k = {"adam": 6, "adagrad": 4, "rmsprop": 6, "sgd": 2}.get(args.learner.lower(), 2)   # var(+slots) read+write
    alg = {   # algorithmic bytes per launch, SURVEY 8(d) (fp32)
        "fwd": B * (28 * D + 16),
        "user_chunk": uniq_users * adam_k * 20 * D,
        "item_chunk": uniq_items * adam_k * 4 * D,
    }
    fused = bool(getattr(eng, "single_pass", False)) and not os.environ.get("FOODREC_TWO_PASS")
    if fused:
        # single-pass step: ONE kernel scores and updates (phase "fwd"; "user_chunk" is the 2 MB commit pass).  Its
        # compulsory bytes: P, m, v read + written once per unique user, the two recipe rows, ids and the two z-stash
        # rows per triple.  SURVEY 8(d) counts the P row once more per triple (its forward figure, 28D+16) on top of
        # the update figure: that sum is reported as survey_alg_bytes, the roofline uses the smaller compulsory figure.
        alg["fwd"] = uniq_users * adam_k * 20 * D + B * (2 * 4 * D + 16) + B * 2 * 4 * D
        alg.pop("user_chunk")
    kern = {k: {"ms": phases[k], "alg_bytes": alg[k], "gbs": alg[k] / (phases[k] * 1e-3) / 1e9 if phases[k] > 0 else None}
            for k in alg}
    if fused:
        kern["fwd"]["survey_alg_bytes"] = B * (28 * D + 16) + uniq_users * adam_k * 20 * D
        kern["fwd"]["gbs_survey"] = kern["fwd"]["survey_alg_bytes"] / (phases["fwd"] * 1e-3) / 1e9
    if args.learner.lower() == "adam" and args.adam_mode != "dense" and not fused:
        # lazy Adam: a user row that was not touched last step is caught up IN REGISTERS before it is scored, which
        # needs its m and v rows too (2 x 20D more bytes per triple; at cfg2 practically every row is stale).  Those
        # reads are compulsory for TF-1.x-exact results without the dense sweep, but are not in SURVEY 8(d)'s figure.
        full = B * (28 * D + 16 + 2 * 20 * D + 2 * 4 * D)          # + m,v rows of P[u] + the two z-stash row writes
        kern["fwd"].update(bytes_incl_adam_state=full, gbs_incl_adam_state=full / (phases["fwd"] * 1e-3) / 1e9,
                           )
    dom = max(alg, key=lambda k: phases[k])
    roofline = {"bound": "hbm", "kernel": {"fwd": "user_fused_kernel" if fused else "fwd_train_kernel", "user_chunk": "seg_chunk_kernel<UserPol>",
                                           "item_chunk": "seg_chunk_kernel<ItemPol>"}[dom],
                "achieved": kern[dom]["gbs"], "peak": peak, "unit": "GB/s", "frac": kern[dom]["gbs"] / peak,
                "peak_source": peak_src, "traffic": None,
                "alg_bytes_per_launch": alg[dom], "ms_per_launch": phases[dom]}
    # dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of each kernel, from the ncu --set full captures of this
    # build (ncu_traffic(): null unless profiles/ncu_traffic.json was made from the sources the library was built from)
    traffic = ncu_traffic()
    kname = {"fwd": "user_fused_kernel" if fused else "fwd_train_kernel", "user_chunk": "seg_chunk_kernel<UserPol>",
             "item_chunk": "seg_chunk_kernel<ItemPol>"}
    for k in kern:
        kern[k]["ncu_dram_bytes_per_launch"] = traffic.get(kname[k])
    roofline["traffic"] = traffic.get(kname[dom])
    # the whole step against the HBM roofline: SURVEY 8(d)'s step total (score + user update + recipe update + G write)
    step_bytes = B * (28 * D + 16) + uniq_users * adam_k * 20 * D + uniq_items * adam_k * 4 * D + 4 * Lb * 5 * D
    roofline_step = {"bound": "hbm", "alg_bytes_per_step": step_bytes, "ms_per_step": ms / args.steps,
                     "achieved": step_bytes / (ms / args.steps * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                     "frac": step_bytes / (ms / args.steps * 1e-3) / 1e9 / peak,
                     "definition": "SURVEY 8(d) train-step total: B(28D+16) + uniq_users*6*20D + uniq_items*6*4D + 4*L*5D bytes"}
    if dom == "fwd" and "gbs_incl_adam_state" in kern["fwd"]:
        roofline["achieved_incl_adam_state"] = kern["fwd"]["gbs_incl_adam_state"]
        roofline["frac_incl_adam_state"] = kern["fwd"]["gbs_incl_adam_state"] / peak
        roofline["note"] = ("achieved/frac use SURVEY 8(d)'s 28D+16 B per triple; the lazy-Adam forward also has to read "
                            "the m and v rows of every stale user row (see kernels.fwd), which the *_incl_adam_state "
                            "figures and the ncu dram traffic include")

    # ---- e2e: reference-format dense feed from pinned host memory through the C ABI host entry point
    pin = lambda x: torch.as_tensor(np.ascontiguousarray(x)).pin_memory()
    hb = [dict(users=pin(b["users"]), items=pin(b["items"]), cats=pin(b["cats"]), ulab=pin(b["ulab"])) for b in host]
    h2d = sum(int(t.numel() * t.element_size()) for t in hb[0].values())

    def estep(k, dense=True):
        b = hb[k % NB]
        return eng.train_step_host(L.FR_BPR, B, b["users"], b["items"], b["cats"] if dense else None, None, None,
                                   b["ulab"] if dense else None)

    def eprefetch(k, dense=True):
        b = hb[k % NB]
        eng.feed_prefetch(L.FR_BPR, B, b["users"], b["items"], b["cats"] if dense else None, None, None,
                          b["ulab"] if dense else None)

    def e2e_run(dense, prefetch=True):
        for k in range(3):
            estep(k, dense)
        barrier()
        t0 = time.perf_counter()
        loss_sum = 0.0
        if prefetch:
            eprefetch(0, dense)
        for k in range(args.steps):
            if prefetch:
                eprefetch(k + 1, dense)                    # H2D of the next feed overlaps this step's kernels
            out = estep(k, dense)
            torch.cuda.current_stream().synchronize()      # the step's loss is read on the host every step
            loss_sum += float(out[L.FR_OUT_LOSS])
        barrier()
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); dt = float(t.item())
        return world * B * args.steps / dt, loss_sum / args.steps
    # the overlapped leg is run three times; the MEDIAN is reported, all three and their spread are in the line
    e2e_run(True)                                  # (untimed: first touch of the staging buffers / copy stream)
    e2e_runs = [e2e_run(True) for _ in range(3)]
    e2e_val, e2e_loss = sorted(e2e_runs)[1]
    e2e_serial, _ = e2e_run(True, prefetch=False)
    e2e_cval, _ = e2e_run(False)

    # ---- pointwise instances/s: the reference's own objective (sigmoid cross-entropy on (user, item, label) rows,
    # Model_Recommender.py:99-104) -- the mode the reference traces pin; same tables, B rows per step, ids resident
    pw = None
    if world == 1:
        rng = np.random.default_rng(77)
        pwb = []
        for k in range(NB):
            pu = torch.as_tensor(rng.integers(0, U, B).astype(np.int32)).to(dev)
            pi = torch.as_tensor(synth.zipf_items(rng, I, B).astype(np.int32)).to(dev)
            py = torch.as_tensor((rng.random(B) < 0.8).astype(np.float32)).to(dev)
            pwb.append((pu, pi, py))

        def pstep(k):
            pu, pi, py = pwb[k % NB]
            eng._step_dev(L.FR_POINTWISE, B, pu, pi, None, py, None, None)
        for k in range(max(args.warmup, 3)):
            pstep(k)
        torch.cuda.synchronize()
        eng.timing_read()
        eng.timing_enable(True)
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record()
        for k in range(args.steps):
            pstep(k)
        p1.record(); torch.cuda.synchronize()
        pph, _ = eng.timing_read()
        eng.timing_enable(False)
        pms = p0.elapsed_time(p1) / args.steps
        pw = {"metric": "pointwise_train_instances_per_sec", "value": B / (pms * 1e-3), "unit": "instances/s",
              "ms_per_step": pms, "batch": B, "phases_ms": pph,
              "fwd_gbs_incl_adam_state": B * (24 * D + 32 + 2 * 20 * D + 4 * D) / (pph["fwd"] * 1e-3) / 1e9 if pph["fwd"] > 0 else None}

    # ---- top-K users/s: sampled evaluation (51 candidates, K=10: evaluate.py) over NU users
    NU = min(U, 1 << 20)
    rng = np.random.default_rng(5)
    eu = torch.as_tensor(rng.permutation(U)[:NU].astype(np.int32)).to(dev)
    cand = torch.as_tensor(rng.integers(0, I, (NU, 51)).astype(np.int32)).to(dev)
    nc = torch.full((NU,), 51, dtype=torch.int32, device=dev)
    eng.eval_sampled_topk(eu, cand, nc, 10)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); eng.eval_sampled_topk(eu, cand, nc, 10); e1.record(); torch.cuda.synchronize()
    eval_ms = e0.elapsed_time(e1)
    eval_alg = NU * (20 * D + 51 * 4 * D + 51 * 12)

    # ---- full-catalog top-100 users/s (tcgen05 GEMM + fused top-K filter): every user of cfg2 on the tables ALL the
    # legs above have trained (pre-roll + timed + per-kernel + e2e + pointwise: several hundred steps, the hot Zipf
    # recipes' norms have grown -- the per-tile filter bound keeps the margin local), then a cfg4-shaped sample (10M
    # recipes) on fresh tables
    catalog = []
    catalog_launches_cfg2 = 0
    if not args.no_catalog:
        lc0 = eng.lib.fr_launch_count()
        catalog.append(bench_catalog(eng, dev, f"cfg2: all {U} users x {I} recipes, D={D}, K=100", U))
        catalog[0]["train_steps_before"] = int(eng.step)
        catalog_launches_cfg2 = eng.lib.fr_launch_count() - lc0
        launches_c0 = eng.lib.fr_launch_count()
        if not args.small:
            eng.close()
            del eng
            torch.cuda.empty_cache()
            # BASELINE configs[3] IN FULL on one GPU: top-100 of 10M recipes for every one of 1M users (14 passes of
            # 75,776 users; one timed run after a one-pass warm-up)
            I4, U4 = 10_000_000, 1_000_000
            g4 = torch.Generator(device=dev); g4.manual_seed(4)
            e4 = Engine(Hyper(learner="sgd"), torch.randn((U4, 5, D), device=dev, generator=g4) * 0.1,
                        torch.randn((I4, D), device=dev, generator=g4) * 0.1, Cat, G, device=dev, max_rows=256,
                        item_cats=synth.make_item_categories(I4), adopt=True)
            catalog.append(bench_catalog(e4, dev, f"cfg4: all {U4} users x {I4} recipes, D={D}, K=100", U4, reps=1,
                                         warm_users=75_776))
            eng = e4
        catalog_launches = catalog_launches_cfg2 + eng.lib.fr_launch_count() - launches_c0

    cfg5 = None
    if world == 1 and not args.no_cfg5:
        cfg5 = cfg5_leg(args, cfg, B, dev, args.steps)
    if rank == 0:
        for tid in os.listdir("/proc/self/task"):          # the CPU legs use every core the box gives us: every thread
            try:                                           # (pool threads created while bound inherited the mask)
                os.sched_setaffinity(int(tid), full_affinity)
            except OSError:
                pass
        cpu = cpu_baseline_leg(cfg, B) if (world == 1 and not args.no_cpu) else None
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(cfg, B), "batch_triples": B, "optimizer": (f"adam (TF-1.x semantics, {args.adam_mode})" if args.learner.lower() == "adam" else args.learner),
                       "l2": "per-step working set (~%.1f GB of table rows) >> 126 MB L2; %d distinct batches cycled" % (
                           sum(alg.values()) / 1e9, NB),
                       "preroll_steps": preroll,
                       "parallelism": "1 GPU" if world == 1 else f"{world} independent replicas (sharded path: see DESIGN.md)"},
            "clocks": clk, "gpu_launches": int(launches),
            "roofline": roofline, "roofline_step": roofline_step, "kernels": kern, "phases_ms": phases,
            "single_pass": fused,
            "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4 * L.FR_OUT_COUNT,
                    "feed": "reference dense feed (user_input,item_input,categories,user_one_hot_label), pinned, "
                            "host read of the loss every step; the copy of feed k+1 (fr_feed_prefetch, library copy "
                            "stream) overlaps the kernels of step k; median of 3 runs of K steps after one untimed run", "mean_loss": e2e_loss,
                    "runs": [v for v, _ in e2e_runs],
                    "spread": (max(v for v, _ in e2e_runs) - min(v for v, _ in e2e_runs)) / e2e_val,
                    "without_prefetch": e2e_serial},
            "e2e_compact": {"value": e2e_cval, "unit": UNIT, "h2d_bytes_per_step": 12 * B,
                            "feed": "ids only; dish_to_category / user labels resident on device"},
            "topk": {"metric": "sampled_topk_users_per_sec", "value": NU / (eval_ms * 1e-3), "unit": "users/s",
                     "candidates": 51, "K": 10, "users": NU, "ms": eval_ms,
                     "roofline": {"bound": "hbm", "achieved": eval_alg / (eval_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                                  "frac": eval_alg / (eval_ms * 1e-3) / 1e9 / peak}},
            "pointwise": pw, "host_numa": numa,
            "uniq_users_per_step": uniq_users, "uniq_items_per_step": uniq_items,
            "cfg5": cfg5,
        }
        if catalog:
            if world == 1 and not args.no_cpu:
                catalog[0]["cpu_baseline"] = cpu_catalog_leg(cfg)
            line["catalog_topk"] = catalog
            line["catalog_gpu_launches"] = int(catalog_launches)
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if world == 1 and not args.no_cpu:
            # BASELINE.md section 3: cfg1 exactly (the reference's own CPU-runnable case), both arms
            line["cfg1"] = {"workload": "cfg1: 10000 users x 5000 recipes x 95 labels, D=64, pointwise B=128, reference stream, Adam",
                            "gpu_e2e": cfg1_gpu_leg(dev), "cpu_baseline": cfg1_cpu_leg()}
        print(json.dumps(line, default=float))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=262144)
    ap.add_argument("--preroll", type=int, default=40)
    ap.add_argument("--small", action="store_true", help="tiny tables: harness check only, not a bench number")
    ap.add_argument("--no-p2p", action="store_true", help="N>1: stage exchanged rows and move them with NCCL all-to-alls instead "
                    "of storing them straight into peer memory (NVLink) from the gather / gradient kernels")
    ap.add_argument("--cfg3", action="store_true", help="100M users / 10M recipes (row-sharded, 8 GPUs: 96 GB of tables+slots per GPU)")
    ap.add_argument("--fixed-tables", action="store_true", help="N>1: cfg2 tables divided over the ranks (round-1 behaviour) "
                    "instead of a cfg2-sized shard per GPU (constant per-GPU work)")
    ap.add_argument("--no-cfg3", action="store_true", help="N=8: skip the cfg3 leg (100M users / 10M recipes)")
    ap.add_argument("--no-plan-ahead", action="store_true", help="N>1: plan every step in sequence instead of one step ahead on a side stream")
    ap.add_argument("--no-cfg5", action="store_true", help="skip the cfg5 leg (1:8 sampled negatives, Adagrad, bf16 tables)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-catalog", action="store_true", help="skip the full-catalog top-K legs")
    ap.add_argument("--learner", default="adam", help="adam (reference default) | adagrad | rmsprop | sgd")
    ap.add_argument("--adam-mode", default="lazy", choices=["lazy", "lazy_exact", "dense"])
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed to "
                    "DIR/<name>.npy (float32, ~30 MB: step scalars, Cat, G, a fixed sample of P and R rows), so that two "
                    "builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs covers the single-process GPU run (--impl ours without torchrun)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    cfg = SMALL if args.small else (CFG3 if args.cfg3 else CFG2)
    if args.cfg3 and int(os.environ.get("WORLD_SIZE", "1")) < 8:
        sys.exit("--cfg3 needs the 8-GPU row-sharded run (torchrun --nproc-per-node 8)")
    if args.impl == "reference":
        run_reference(args, cfg, args.batch)
    elif int(os.environ.get("WORLD_SIZE", "1")) > 1:
        run_sharded(args, cfg, args.batch)
    else:
        run_ours(args, cfg, args.batch)


if __name__ == "__main__":
    main()
