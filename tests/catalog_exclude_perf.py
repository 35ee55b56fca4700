"""Perf harness for full-catalog top-K with exclusion lists (not collected by pytest).

cfg2 in full (1M users x 200k recipes, D=128), K = 10 and 100.  Per case: device time per call (CUDA events, one
warm-up call first), the catalog phase times, fr_catalog_fallback_rows of the last pass, and for 256 sampled users
equality with tests/catalog_exclude_oracle.py.  Cases: the plain call (fr_catalog_topk), the new entry
with empty lists, Zipf(1.05) histories of 20 and of 50 recipes per user (drawn like bench.py's positives), and a mix
where 1 % of the users have 400 seen recipes (the others 20).

    python tests/catalog_exclude_perf.py [--reps 5] [--parent-lib PATH] [--out FILE]

--parent-lib: a library built from the parent commit's sources, e.g. in a checkout of that commit
    python -c "from foodrec_b200 import _build; _build.build_variant('parent', [])"
(-> foodrec_b200/csrc/libfoodrec_b200_parent.so there).  The plain cfg2 call is then timed A/B, alternating this
build and the parent build in fresh processes (FOODREC_B200_LIB selects the library of a process)."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import synth_data as synth  # noqa: E402

U, I, D = 1_000_000, 200_000, 128


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def make_engine(seed=11):
    from foodrec_b200 import Engine, Hyper
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev); g.manual_seed(seed)
    P = torch.randn((U, 5, D), generator=g, device=dev) * 0.1
    R = torch.randn((I, D), generator=g, device=dev) * 0.1
    Cat = torch.randn((4, D), generator=g, device=dev) * 0.1
    ic = synth.make_item_categories(I, seed=seed + 1)
    e = Engine(Hyper(), P, R, Cat, torch.zeros((9, 5, D), device=dev), max_rows=256, item_cats=ic, adopt=True)
    e.catalog_prepare()
    return e, ic


def histories(kind, seed=5):
    """CSR (offsets [U+1], ids) of the seen lists of every user."""
    rng = np.random.default_rng(seed)
    if kind == "empty":
        return np.zeros(U + 1, np.int32), np.zeros(0, np.int32)
    if kind in ("zipf20", "zipf50"):
        lens = np.full(U, int(kind[4:]), np.int64)
    else:                                                    # heavy: 1 % of the users have seen 400 recipes
        lens = np.full(U, 20, np.int64)
        lens[rng.choice(U, U // 100, replace=False)] = 400
    off = np.zeros(U + 1, np.int64); off[1:] = np.cumsum(lens)
    return off.astype(np.int32), synth.zipf_items(rng, I, int(off[-1]))


def time_calls(e, K, excl, reps):
    """ms per call (CUDA events), phase ms per call, fallback rows, last result."""
    e.timing_enable(True)
    ids, sc = e.catalog_topk(n_users=U, K=K, exclude=excl)     # warm-up (workspace, code load)
    torch.cuda.synchronize(); e.catalog_timing_read()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); ids, sc = e.catalog_topk(n_users=U, K=K, exclude=excl); b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    ph, passes = e.catalog_timing_read()
    e.timing_enable(False)
    return ms, {k: v / reps for k, v in ph.items()}, e.catalog_fallback_rows(), ids, sc


def oracle_check(e, ic, K, ids, sc, excl, n=256, seed=1):
    from oracle import evaluate_oracle
    from tests import catalog_exclude_oracle as xo
    from oracle.recommender_oracle import Hyper as OHyper, OracleModel
    rng = np.random.default_rng(seed)
    sample = np.sort(rng.choice(U, n, replace=False))
    ts = torch.as_tensor(sample).to(e.device)
    om = OracleModel(e.P[ts].cpu().numpy(), e.R.cpu().numpy(), e.Cat.cpu().numpy(), np.zeros((9, 5, D), np.float32),
                     OHyper(), dtype=np.float32)
    ex = None if excl is None else [excl[1][excl[0][u]:excl[0][u + 1]] for u in sample]
    rid, rsc = (evaluate_oracle.catalog_topk(om, np.arange(n), ic, K) if ex is None
                else xo.catalog_topk_excluding(om, np.arange(n), ic, K, ex))
    gi, gs = ids[ts].cpu().numpy(), sc[ts].cpu().numpy()
    fin = np.isfinite(rsc)
    return bool(np.array_equal(gi, rid) and np.array_equal(fin, np.isfinite(gs))
                and np.abs(gs[fin] - rsc[fin]).max() <= 1e-12 * np.abs(rsc[fin]).max())


def cases(reps, out):
    e, ic = make_engine()
    lists = {k: histories(k) for k in ("empty", "zipf20", "zipf50", "heavy")}
    # resident device CSR: the timed window holds the call, not the host -> device copy of the lists
    dlists = {k: tuple(torch.as_tensor(x).to(e.device) for x in v) for k, v in lists.items()}
    res = []
    for K in (10, 100):
        base = None
        for name in ("plain", "empty", "zipf20", "zipf50", "heavy"):
            excl = None if name == "plain" else lists[name]
            ms, ph, fb, ids, sc = time_calls(e, K, None if excl is None else dlists[name], reps)
            ok = oracle_check(e, ic, K, ids, sc, excl)
            med = float(np.median(ms))
            base = med if name == "plain" else base
            r = {"K": K, "case": name, "ms_median": med, "ms": [round(x, 3) for x in ms], "x_plain": med / base,
                 "phases_ms": {k: round(v, 3) for k, v in ph.items()}, "fallback_rows_last_pass": fb,
                 "oracle_256_users_equal": ok,
                 "list_entries": 0 if excl is None else int(excl[1].size)}
            print(json.dumps(r), flush=True)
            res.append(r)
            del ids, sc
    e.close()
    return res


def plain_only(reps):
    from foodrec_b200 import _lib
    if os.environ.get("CATALOG_PERF_PARENT"):    # the parent library predates the exclusion entry; the plain call needs none
        _lib._PROTOS.pop("fr_catalog_topk_excluding", None)
    e, _ = make_engine()
    for K in (10, 100):
        ms, ph, fb, _, _ = time_calls(e, K, None, reps)
        print("PLAIN " + json.dumps({"K": K, "ms": ms, "phases_ms": ph, "fallback": fb}), flush=True)
    e.close()


def ab(parent_lib, reps, rounds=3):
    from foodrec_b200 import _build
    libs = {"this": _build.LIB, "parent": os.path.abspath(parent_lib)}
    out = {k: {10: [], 100: []} for k in libs}
    phases = {k: {10: [], 100: []} for k in libs}
    for rnd in range(rounds):
        for name in (("this", "parent") if rnd % 2 == 0 else ("parent", "this")):
            env = dict(os.environ, FOODREC_B200_LIB=libs[name])
            if name == "parent":
                env["CATALOG_PERF_PARENT"] = "1"
            p = subprocess.run([sys.executable, os.path.abspath(__file__), "--plain-only", "--reps", str(reps)],
                               capture_output=True, text=True, env=env)
            lines = [json.loads(l[6:]) for l in p.stdout.splitlines() if l.startswith("PLAIN ")]
            if p.returncode != 0 or len(lines) != 2:
                raise RuntimeError(f"{name}: " + p.stdout[-1000:] + p.stderr[-2000:])
            for r in lines:
                out[name][r["K"]] += r["ms"]
                phases[name][r["K"]].append(r["phases_ms"])
    res = []
    for K in (10, 100):
        a, b = np.array(out["this"][K]), np.array(out["parent"][K])
        r = {"ab_plain_call": True, "K": K, "this_median_ms": float(np.median(a)), "parent_median_ms": float(np.median(b)),
             "this_ms": [round(x, 3) for x in a], "parent_ms": [round(x, 3) for x in b],
             "ratio": float(np.median(a) / np.median(b)),
             "phases_ms": {n: {k: round(float(np.median([p[k] for p in phases[n][K]])), 3) for k in phases[n][K][0]}
                           for n in libs}}
        print(json.dumps(r), flush=True)
        res.append(r)
    return res


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--out", default=None)
    ap.add_argument("--ab-only", action="store_true", help="skip the cases, time the plain call A/B only")
    ap.add_argument("--plain-only", action="store_true")
    a = ap.parse_args()
    if a.plain_only:
        plain_only(a.reps)
        sys.exit(0)
    info = gpu_info()
    print("GPU (name, power limit, max SM clock):", info, flush=True)
    res = {"gpu": info, "cfg": f"{U} users x {I} recipes, D={D}", "cases": [] if a.ab_only else cases(a.reps, a.out)}
    if a.parent_lib:
        res["ab"] = ab(a.parent_lib, a.reps)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
