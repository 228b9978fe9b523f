"""A/B of the double-hoisted rotate-multiply-sum (Evaluator.rotate_multiply_sum_hoisted) against the modes it competes with,
in one process, alternating the variants of a workload `--reps` times, each call timed with CUDA events:

  config 3 (N = 16384, {60, 40, 40, 60}), d = 64 and 128:  Linear_Transform_Plain (bit-identical), hoisted, BSGS + hoisted,
                                                           double-hoisted, BSGS double-hoisted
  config 4 (N = 16384, {60, 40 x 4, 60}), d = 64:          cc_matrix_multiplication_nonzero against _nonzero_hoisted

Per variant: the median time, the max decrypted error against the plaintext result, the key inner products and mod-downs
per call (counted from the plans, the duplicate fill's rotation included) and memory: torch's peak allocation (keys,
plaintexts, ciphertexts) and the device memory in use after the variant (that also holds the engine's workspace).

usage: python profiles/double_hoisting_ab.py [--out FILE.json] [--reps 5]
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


def gpu_info():
    q = ["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"]
    try:
        return subprocess.run(q, stdout=subprocess.PIPE, text=True, timeout=60).stdout.strip().splitlines()
    except (OSError, subprocess.SubprocessError) as e:
        return ["unavailable: %s" % e]


def timed(torch, fn, reps_out):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    res = fn()
    e1.record()
    torch.cuda.synchronize()
    reps_out.append(e0.elapsed_time(e1))
    return res


def run_variants(torch, variants, reps, err_of):
    """variants: name -> (fn, counts); alternated reps times after one warm-up call each"""
    out = {}
    for name, (fn, counts) in variants.items():
        torch.cuda.reset_peak_memory_stats()
        err = err_of(fn())
        torch.cuda.synchronize()
        free, total = torch.cuda.mem_get_info()
        out[name] = dict(counts, max_err=float(err), ms=[], torch_peak_mb=round(torch.cuda.max_memory_allocated() / 2 ** 20, 1),
                         device_used_mb=round((total - free) / 2 ** 20, 1))
    for _ in range(reps):
        for name, (fn, _) in variants.items():
            timed(torch, fn, out[name]["ms"])
    for v in out.values():
        v["median_ms"] = round(statistics.median(v["ms"]), 3)
        v["ms"] = [round(x, 3) for x in v["ms"]]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    import numpy as np
    import torch
    assert torch.cuda.is_available(), "this measurement needs a CUDA device"
    eng = importlib.import_module(PKG).load_engine()
    wl = importlib.import_module(PKG + ".workloads")
    client = importlib.import_module(PKG + ".client")
    params = importlib.import_module(PKG + ".params")
    rec = {"gpu": gpu_info(), "reps": a.reps, "workloads": {}}
    scale = 2.0 ** 40

    # ---- config 3: linear transforms
    ctx = eng.Context(14, params.coeff_modulus_create(14, [60, 40, 40, 60]))
    ev, enc = eng.Evaluator(ctx), client.CKKSEncoder(ctx)
    kg = client.KeyGenerator(ctx, seed=5)
    steps = set()
    for d in (64, 128):
        steps |= set(wl.linear_transform_double_hoisted_steps(d))
    keys = kg.keyset(steps=sorted(steps), relin=False)
    key_mb = len(keys.galois) * (ctx.K - 1) * 2 * ctx.K * ctx.n * 8 / 2 ** 20
    encr, decr = client.Encryptor(ctx, kg.public_key(), seed=6), client.Decryptor(ctx, kg.secret_key())
    plans = wl.PlanCache(ctx, keys)
    for d in (64, 128):
        rng = np.random.default_rng(d)
        U, v = rng.uniform(0, 1, (d, d)), rng.uniform(0, 1, d)
        want = U @ v
        ct = encr.encrypt(enc.encode(v, scale))
        diags = enc.encode(wl.all_diagonals(U), scale)
        diags_k = enc.encode(wl.all_diagonals(U), scale, limbs=ctx.K)
        bd, bd_k = wl.BsgsDiagonals(U, scale, enc), wl.BsgsDiagonals(U, scale, enc, limbs=ctx.K)
        b, G = bd.b, bd.G
        lt = plans.rms(1, d, wl.diagonal_terms([range(d)], [0]))
        baby, giant = wl.bsgs_terms(d, b)
        pb, pg = plans.rms(1, d, baby), plans.rms(G, 0, giant)
        shared = plans.get(range(d)).keyswitches_shared
        c = lambda ip, md: {"inner_products": ip, "mod_downs": md}
        variants = {
            "bit_identical": (lambda: wl.linear_transform_plain(ev, ct, diags, keys, plans), c(1 + shared, 1 + shared)),
            "hoisted": (lambda: wl.linear_transform_plain_hoisted(ev, ct, diags, keys, plans), c(d, d)),
            "bsgs_hoisted": (lambda: wl.linear_transform_plain_bsgs_hoisted(ev, ct, bd, keys, plans), c(b + G - 1, b + G - 1)),
            "double_hoisted": (lambda: wl.linear_transform_plain_double_hoisted(ev, ct, diags_k, keys, plans),
                               c(1 + lt.inner_products, 1 + lt.mod_downs)),
            "bsgs_double_hoisted": (lambda: wl.linear_transform_plain_bsgs_double_hoisted(ev, ct, bd_k, keys, plans),
                                    c(1 + pb.inner_products + pg.inner_products, 1 + pb.mod_downs + pg.mod_downs)),
        }
        err = lambda x: np.abs(enc.decode(decr.decrypt(x))[0, :d] - want).max()
        rec["workloads"]["config3_d%d" % d] = {"baby": b, "giants": G, "keys": len(keys.galois), "keys_mb": round(key_mb, 1),
                                               "variants": run_variants(torch, variants, a.reps, err)}
        print(json.dumps(rec["workloads"]["config3_d%d" % d]), flush=True)
    del keys, plans, ctx, ev, enc, kg
    torch.cuda.empty_cache()

    # ---- config 4: the 64 x 64 product
    d = 64
    dd = d * d
    ctx = eng.Context(14, params.coeff_modulus_create(14, [60, 40, 40, 40, 40, 60]))
    ev, enc = eng.Evaluator(ctx), client.CKKSEncoder(ctx)
    kg = client.KeyGenerator(ctx, seed=7)
    keys = kg.keyset(steps=wl.matmul_nonzero_hoisted_steps(d))
    key_mb = len(keys.galois) * (ctx.K - 1) * 2 * ctx.K * ctx.n * 8 / 2 ** 20
    encr, decr = client.Encryptor(ctx, kg.public_key(), seed=8), client.Decryptor(ctx, kg.secret_key())
    plans = wl.PlanCache(ctx, keys)
    rng = np.random.default_rng(dd)
    A, B = rng.uniform(0, 1, (d, d)), rng.uniform(0, 1, (d, d))
    ctA, ctB = encr.encrypt(enc.encode(A.reshape(-1), scale)), encr.encrypt(enc.encode(B.reshape(-1), scale))
    both = lambda U: (wl.DiagonalSet.from_matrix(U, 1e-8, scale, enc), wl.DiagonalSet.from_matrix(U, 1e-8, scale, enc, limbs=ctx.K))
    sig, tau = both(wl.u_sigma(d)), both(wl.u_tau(d))
    V = [both(wl.v_k(d, k)) for k in range(1, d)]
    W = [both(wl.w_k(d, k)) for k in range(1, d)]
    first, second = wl.matmul_nonzero_hoisted_terms(sig[1].index, tau[1].index, [s[1].index for s in V], [s[1].index for s in W])
    n1 = len(sig[1].index) + len(tau[1].index)
    p1, p2 = plans.rms(2, n1, first), plans.rms(2, sum(len(t) for t in second), second)
    steps2 = lambda sets: plans.get(sorted({l for s in sets for l in s.index})).keyswitches_shared
    ks_nz = 4 + plans.get(sig[0].index).keyswitches_shared + plans.get(tau[0].index).keyswitches_shared + \
        steps2([v[0] for v in V]) + steps2([w[0] for w in W])
    c = lambda ip, md: {"inner_products": ip, "mod_downs": md}
    variants = {
        "nonzero": (lambda: wl.cc_matrix_multiplication_nonzero(ev, ctA, ctB, d, sig[0], tau[0], [v[0] for v in V],
                                                                [w[0] for w in W], keys, plans), c(ks_nz, ks_nz)),
        "nonzero_hoisted": (lambda: wl.cc_matrix_multiplication_nonzero_hoisted(ev, ctA, ctB, d, sig[1], tau[1], [v[1] for v in V],
                                                                                [w[1] for w in W], keys, plans),
                            c(4 + p1.inner_products + p2.inner_products, 4 + p1.mod_downs + p2.mod_downs)),
    }
    want = A @ B
    err = lambda x: np.abs(enc.decode(decr.decrypt(x))[0, :dd].reshape(d, d) - want).max()
    rec["workloads"]["config4_matmul_d64"] = {"keys": len(keys.galois), "keys_mb": round(key_mb, 1),
                                              "variants": run_variants(torch, variants, a.reps, err)}
    print(json.dumps(rec["workloads"]["config4_matmul_d64"]), flush=True)
    text = json.dumps(rec, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
