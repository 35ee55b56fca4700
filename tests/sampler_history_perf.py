"""Cost of rejecting each user's history in the negative sampler (not collected by pytest):

    python tests/sampler_history_perf.py [--reps 11] [--out FILE]

cfg5 sizes (1M users, 200k recipes, 32,768 positives x 8 negatives = 262,144 draws per step).  Histories: recipes drawn
Zipf(1.05), row lengths geometric with a mean of 20, of 50, and mean 20 with 1 % of the users holding 400.  Reported in
one JSON line, every figure as {median, min, max} over ``reps`` windows, the variants alternating window by window:
  * the sampler alone (fr_sample_batch, FR_SAMPLE_BPR layout), us per call of 262,144 draws, without a history and with
    each of the three: the kernel's own duration (torch.profiler, 200 calls per variant), and the calls through
    Engine.sample_bpr_batch between two CUDA events (200 per window; this one includes the Python and launch overhead
    that bounds a lone call);
  * the cfg5 one-GPU step (bf16 tables, Adagrad, D = 128: bench.py's cfg5 leg) via Engine.train_step_sampled, ms per
    step with and without exclude_seen (mean-20 histories); a window is 20 steps;
  * the card and its power limit, read in the same run."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

U, I, LB, D, N_POS, N_NEG = 1_000_000, 200_000, 95, 128, 32768, 8


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def history(rng, mean, heavy=0.0, heavy_len=400):
    import synth_data
    lens = rng.geometric(1 / mean, U)
    if heavy:
        lens[rng.random(U) < heavy] = heavy_len
    off = np.zeros(U + 1, np.int64); off[1:] = np.cumsum(lens)
    key = np.repeat(np.arange(U, dtype=np.int64), lens) * I + synth_data.zipf_items(rng, I, int(off[-1]))
    key.sort()                                          # rows ascending
    ids = key % I
    return (torch.as_tensor(off.astype(np.int32)).cuda(), torch.as_tensor(ids.astype(np.int32)).cuda()), int(off[-1])


def stats(xs):
    return {"median": float(np.median(xs)), "min": float(np.min(xs)), "max": float(np.max(xs))}


def windows(variants, per_window, reps):
    """{name: [ms per call of each window]}: the variants run alternately, window by window."""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    out = {k: [] for k in variants}
    for _ in range(reps):
        for name, (setup, fn) in variants.items():
            setup()
            torch.cuda.synchronize()
            a.record()
            for k in range(per_window):
                fn(k)
            b.record(); torch.cuda.synchronize()
            out[name].append(a.elapsed_time(b) / per_window)
    return out


def kernel_us(setup, fn, calls):
    """Durations (us) of the sampler kernel over ``calls`` calls, from a torch.profiler trace."""
    import tempfile
    from torch.profiler import ProfilerActivity, profile
    setup()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for k in range(calls):
            fn(k)
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            ev = json.load(f)["traceEvents"]
    return [e["dur"] for e in ev if e.get("cat") == "kernel" and "sample_kernel" in e.get("name", "")]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=11)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from foodrec_b200 import Engine, Hyper
    import synth_data
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(5)
    hists = {"mean20": history(rng, 20), "mean50": history(rng, 50), "mean20_1pct_400": history(rng, 20, heavy=0.01)}
    NB = 8
    batches = [(torch.as_tensor(rng.integers(0, U, N_POS).astype(np.int32)).cuda(),
                torch.as_tensor(synth_data.zipf_items(rng, I, N_POS).astype(np.int32)).cuda()) for _ in range(NB)]
    res = {"users": U, "recipes": I, "draws_per_call": N_POS * N_NEG,
           "history_ids": {k: n for k, (_, n) in hists.items()}}

    # the sampler alone
    g = torch.Generator(device=dev); g.manual_seed(5)
    eng = Engine(Hyper(learner="adagrad", lr=0.01), torch.zeros((U, 5, 4), device=dev), torch.zeros((I, 4), device=dev),
                 torch.zeros((4, 4), device=dev), torch.zeros((3, 5, 4), device=dev), device=dev, max_rows=256, adopt=True)

    def draw(ex):
        return lambda k: eng.sample_bpr_batch(*batches[k % NB], N_NEG, seed=20260105, sample_offset=k * N_POS, exclude_seen=ex)
    variants = {"none": (lambda: None, draw(False))}
    for name, (h, _) in hists.items():
        variants[name] = ((lambda h=h: eng.set_user_history(h)), draw(True))
    for name, (setup, fn) in variants.items():          # warm-up
        setup(); fn(0)
    w = windows(variants, 200, args.reps)
    res["sampler_call_us"] = {k: stats(np.array(v) * 1e3) for k, v in w.items()}
    res["sampler_kernel_us"] = {k: stats(kernel_us(setup, fn, 200)) for k, (setup, fn) in variants.items()}
    eng.close(); del eng

    # the cfg5 one-GPU step: bf16 tables, Adagrad
    item_cats = synth_data.make_item_categories(I)
    lab = synth_data.make_user_label_csr(U, LB)
    P = (torch.randn((U, 5, D), device=dev, generator=g) * 0.1).to(torch.bfloat16)
    R = (torch.randn((I, D), device=dev, generator=g) * 0.1).to(torch.bfloat16)
    Cat = torch.randn((4, D), device=dev, generator=g) * 0.1; G = torch.randn((LB, 5, D), device=dev, generator=g) * 0.1
    eng = Engine(Hyper(learner="adagrad", lr=0.01), P, R, Cat, G, device=dev, max_rows=2 * N_POS * N_NEG, item_cats=item_cats,
                 user_label_csr=lab, adopt=True, table_dtype="bf16")
    del P, R
    eng.set_user_history(hists["mean20"][0])

    def step(ex):
        return lambda k: eng.train_step_sampled(*batches[k % NB], N_NEG, seed=20260105, sample_offset=k * N_POS, exclude_seen=ex)
    sv = {"plain": (lambda: None, step(False)), "exclude_seen": (lambda: None, step(True))}
    for _, fn in sv.values():
        for k in range(10):
            fn(k)
    eng.read_scalars()
    w = windows(sv, 20, args.reps)
    res["cfg5_step_ms"] = {k: stats(v) for k, v in w.items()}
    res["cfg5_step_extra_us_median"] = (np.median(w["exclude_seen"]) - np.median(w["plain"])) * 1e3
    eng.read_scalars()
    eng.close()
    res["gpu"] = gpu_info()
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
