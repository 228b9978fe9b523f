"""A/B of the rotate-and-sum chain step: the product library (c0 carried split, 17 instead of 20 transforms per step at
L = 3) against a baseline build of the same sources with -DV_CHAIN_NOSPLIT (every step transforms c0's mod-down remainder,
the chain of the parent revision).  Each library runs in a process of its own (CKKS_B200_LIB), alternating product and
baseline three times; each process times every shape with CUDA events around a long graph-replayed chain.

usage: profiles/build_variant.sh nosplit -DV_CHAIN_NOSPLIT
       python profiles/chain_split_ab.py [--variant profiles/variants/libckks_nosplit.so] [--out FILE.json] [--rounds 3]
"""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = "seal-fyp-logistic-regression_b200"
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
# (L, batch): the bench chain's level at the batches of 1 to 8 GPUs and below, and the top of the chain
SHAPES = [(3, 32), (3, 16), (3, 8), (3, 4), (3, 2), (3, 1), (9, 32)]
STEPS = 200     # dependent steps per timed call (per lane 12 graph launches of 8 pairs and 4 of 1 pair, then the fold)


def child():
    import torch
    pkg = importlib.import_module(PKG)
    eng = pkg.load_engine()
    params = importlib.import_module(PKG + ".params")
    client = importlib.import_module(PKG + ".client")
    primes = params.coeff_modulus_create(15, [60] + [40] * 8 + [60])
    ctx = eng.Context(15, primes)
    ev = eng.Evaluator(ctx)
    keys = client.KeyGenerator(ctx, seed=1).keyset(steps=[1])
    out = {}
    for L, batch in SHAPES:
        gen = torch.Generator(device="cuda").manual_seed(77 + L + batch)
        dup = ctx.empty(batch, 2, L, cap=9)
        dup.data.random_(0, 1 << 39, generator=gen)
        acc, scratch = dup.clone(), dup.like()
        run = lambda: ev.rotate_sum_chain(dup, acc, 1, STEPS, keys, scratch=scratch)
        run()   # graph capture, allocation
        torch.cuda.synchronize()
        reps = 3 if L == 3 else 1
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            run()
        e1.record()
        torch.cuda.synchronize()
        out["L%d_b%d" % (L, batch)] = e0.elapsed_time(e1) / reps / STEPS * 1e3   # us per chain step
    print("RESULT " + json.dumps(out), flush=True)


def gpu_info():
    q = ["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"]
    try:
        return subprocess.run(q, stdout=subprocess.PIPE, text=True, timeout=60).stdout.strip().splitlines()
    except (OSError, subprocess.SubprocessError) as e:
        return ["unavailable: %s" % e]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--variant", default=os.path.join(ROOT, "profiles", "variants", "libckks_nosplit.so"))
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--child", action="store_true")
    a = ap.parse_args()
    if a.child:
        return child()
    product = importlib.import_module(PKG + "._build").build()
    libs = {"product": product, "nosplit": os.path.abspath(a.variant)}
    runs = {k: [] for k in libs}
    for r in range(a.rounds):
        for name, lib in libs.items():
            env = dict(os.environ, CKKS_B200_LIB=lib)
            res = subprocess.run([sys.executable, os.path.abspath(__file__), "--child"], env=env, cwd=ROOT,
                                 stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
            line = [x for x in res.stdout.splitlines() if x.startswith("RESULT ")]
            if res.returncode != 0 or not line:
                sys.exit("%s failed:\n%s" % (name, res.stdout[-3000:]))
            runs[name].append(json.loads(line[0][7:]))
            print(name, r, line[0][7:], flush=True)
    summary = {}
    for shape in runs["product"][0]:
        p = [x[shape] for x in runs["product"]]
        b = [x[shape] for x in runs["nosplit"]]
        summary[shape] = {"product_us": [round(v, 2) for v in p], "nosplit_us": [round(v, 2) for v in b],
                          "product_median": round(statistics.median(p), 2), "nosplit_median": round(statistics.median(b), 2),
                          "speedup": round(statistics.median(b) / statistics.median(p), 4)}
    rec = {"what": "rotate-and-sum chain step, us (N = 32768, chain {60, 40 x 8, 60}, %d steps per call)" % STEPS,
           "gpu": gpu_info(), "rounds": a.rounds, "shapes": summary}
    text = json.dumps(rec, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
