"""The blocked encrypted matrix product (workloads.cc_matrix_multiplication_blocked) against the naive loop of per-tile
products, and its contraction kernel (ckks_multiply_sum_matrix) against t grouped calls, in one process on one GPU.

Config-4 chain {60, 40 x 4, 60} at N = 16384, d = 64 tiles (d^2 = N/4):
  hoisted method   at 128 x 128 and 256 x 256: blocked vs sum over l of cc_matrix_multiplication_nonzero_hoisted
  reference method at 128 x 128:               blocked vs sum over l of cc_matrix_multiplication_sparse
The two variants of a workload alternate `--reps` times after one warm-up call each, every call timed with CUDA events;
their outputs are compared word for word.  Per variant: the times, the max decrypted error against A B, torch's peak
memory and the key switches / key inner products per call (counted from the plans: the duplicate fills, the rotation
plans of the reference path and the rotate-multiply-sum tables of the hoisted path).

Contraction: multiply_sum_matrix of the 256 x 256 product's entries (t_n x t_m d by t_m d x t_p at L - 1 = 4 limbs)
against t_p multiply_sum_grouped calls over B's columns gathered beforehand; algorithmic bytes (a and b read once, out
written once) over the kernel time, as a fraction of the 7.7 TB/s HBM3e figure of the B200 data sheet.  The entries
(about 2 GB) do not fit the 126 MB L2.

usage: python profiles/matmul_blocked.py --out-dir DIR [--reps 3]
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
HBM_TBS = 7.7


def gpu_info():
    q = ["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"]
    try:
        return subprocess.run(q, stdout=subprocess.PIPE, text=True, timeout=60).stdout.strip().splitlines()
    except (OSError, subprocess.SubprocessError) as e:
        return ["unavailable: %s" % e]


def timed(torch, fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    res = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out-dir", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--sizes", default="128,256", help="matrix sizes of the hoisted method")
    ap.add_argument("--reference-size", type=int, default=128, help="matrix size of the reference method (0: skip)")
    a = ap.parse_args()
    import numpy as np
    import torch
    assert torch.cuda.is_available(), "this measurement needs a CUDA device"
    eng = importlib.import_module(PKG).load_engine()
    wl = importlib.import_module(PKG + ".workloads")
    client = importlib.import_module(PKG + ".client")
    params = importlib.import_module(PKG + ".params")
    rec = {"gpu": gpu_info(), "reps": a.reps, "chain": [60, 40, 40, 40, 40, 60], "log_n": 14, "d": 64, "workloads": {}}
    scale, eps, d = 2.0 ** 40, 1e-8, 64
    dd = d * d
    ctx = eng.Context(14, params.coeff_modulus_create(14, rec["chain"]))
    ev, enc = eng.Evaluator(ctx), client.CKKSEncoder(ctx)
    kg = client.KeyGenerator(ctx, seed=11)
    pow2 = [s for i in range(13) for s in (1 << i, -(1 << i))]
    keys = {"hoisted": kg.keyset(steps=wl.matmul_nonzero_hoisted_steps(d)), "reference": kg.keyset(steps=pow2)}
    plans = {k: wl.PlanCache(ctx, v) for k, v in keys.items()}
    encr, decr = client.Encryptor(ctx, kg.public_key(), seed=12), client.Decryptor(ctx, kg.secret_key())
    mats = {"hoisted": [], "reference": []}
    for U in [wl.u_sigma(d), wl.u_tau(d)] + [wl.v_k(d, k) for k in range(1, d)] + [wl.w_k(d, k) for k in range(1, d)]:
        mats["reference"].append(wl.DiagonalSet.from_matrix(U, eps, scale, enc))
        mats["hoisted"].append(wl.DiagonalSet.from_matrix(U, eps, scale, enc, limbs=ctx.K))
    args = {m: (v[0], v[1], v[2:d + 1], v[d + 1:], keys[m], plans[m]) for m, v in mats.items()}

    def per_tile_counts(method):
        """(key switches, key inner products) of the operand side of one tile, per side (A, B)"""
        sig, tau, V, W = args[method][:4]
        if method == "reference":
            ks = 2 * (1 + plans[method].get(range(dd)).keyswitches_shared)     # duplicate fill + shared rotations, twice
            return (ks, ks), (ks, ks)
        out = []
        for first, sets in ((sig, V), (tau, W)):
            t1 = plans[method].rms(1, len(first.index), [[(0, l, i) for i, l in enumerate(first.index)]])
            off, t2 = 0, []
            for s in sets:
                t2.append([(0, l, off + i) for i, l in enumerate(s.index)])
                off += len(s.index)
            p2 = plans[method].rms(1, off, t2)
            ip = 2 + t1.inner_products + p2.inner_products                       # + the two duplicate fills
            out.append((2 + t1.mod_downs + p2.mod_downs, ip))
        return tuple(out)

    def run(method, size):
        rng = np.random.default_rng(size)
        A, B = rng.uniform(0, 1, (size, size)), rng.uniform(0, 1, (size, size))
        tA, (tn, tm) = wl.matrix_tiles(A, d)
        tB, (_, tp) = wl.matrix_tiles(B, d)
        At, Bt = encr.encrypt(enc.encode(tA, scale)), encr.encrypt(enc.encode(tB, scale))
        tiles = (tn, tm, tp)
        fn = wl.cc_matrix_multiplication_sparse if method == "reference" else wl.cc_matrix_multiplication_nonzero_hoisted

        def naive():
            outs = []
            for i in range(tn):
                for j in range(tp):
                    acc = None
                    for l in range(tm):
                        p = fn(ev, At[i * tm + l], Bt[l * tp + j], d, *args[method])
                        acc = p if acc is None else ev.add(acc, p)
                    outs.append(acc.data[:, :, :acc.limbs])
            return eng.Ciphertext(ctx, torch.cat(outs), acc.limbs, acc.scale)

        def blocked():
            return wl.cc_matrix_multiplication_blocked(ev, At, Bt, tiles, d, *args[method], method=method)
        (ksA, ipA), (ksB, ipB) = per_tile_counts(method)
        counts = {"blocked": (tn * tm * ksA + tm * tp * ksB, tn * tm * ipA + tm * tp * ipB),
                  "naive": (tn * tm * tp * (ksA + ksB), tn * tm * tp * (ipA + ipB))}
        res = {}
        outs = {}
        for name, f in (("blocked", blocked), ("naive", naive)):
            torch.cuda.synchronize()
            torch.cuda.reset_peak_memory_stats()
            outs[name] = f()
            torch.cuda.synchronize()
            got = wl.matrix_from_tiles(enc.decode(decr.decrypt(outs[name])), (size, size), d)
            key = "keyswitches" if method == "reference" else "mod_downs"
            res[name] = {"ms": [], key: counts[name][0], "inner_products": counts[name][1],
                         "max_err": float(np.abs(got - A @ B).max()),
                         "torch_peak_mb": round(torch.cuda.max_memory_allocated() / 2 ** 20, 1)}
        b, n = outs["blocked"], outs["naive"]
        equal = bool(b.scale == n.scale and b.limbs == n.limbs and torch.equal(b.data[:, :, :b.limbs], n.data[:, :, :n.limbs]))
        del outs
        for _ in range(a.reps):
            for name, f in (("blocked", blocked), ("naive", naive)):
                ms, out = timed(torch, f)
                res[name]["ms"].append(round(ms, 3))
                del out
        for v in res.values():
            v["median_ms"] = round(statistics.median(v["ms"]), 3)
        w = {"tiles": list(tiles), "word_for_word_equal": equal, "variants": res,
             "speedup": round(res["naive"]["median_ms"] / res["blocked"]["median_ms"], 2)}
        rec["workloads"]["%s_%dx%d" % (method, size, size)] = w
        print(json.dumps(w), flush=True)
        torch.cuda.empty_cache()

    for size in [int(s) for s in a.sizes.split(",") if s]:
        run("hoisted", size)
    if a.reference_size:
        run("reference", a.reference_size)

    # ---- the contraction alone, at the 256 x 256 product's shape
    t = 4
    rows, inner, cols, L = t, t * d, t, ctx.K - 2
    g = torch.Generator(device=ctx.device).manual_seed(3)

    def rand(batch):
        ct = ctx.empty(batch, 2, L)
        for j in range(L):
            ct.data[:, :, j].random_(0, ctx.primes[j], generator=g)
        return ct
    X, Y = rand(rows * inner), rand(inner * cols)
    colsY = [eng.Ciphertext(ctx, Y.data[j::cols].contiguous(), L) for j in range(cols)]
    mat = lambda: ev.multiply_sum_matrix(X, Y, rows, cols)
    grouped = lambda: [ev.multiply_sum_grouped(X, colsY[j], rows) for j in range(cols)]
    m, gr = mat(), grouped()
    equal = all(torch.equal(m.data[j::cols], gr[j].data) for j in range(cols))
    reps = max(10, 5 * a.reps)
    times = {"matrix": [], "grouped": []}
    for _ in range(reps):
        for name, f in (("matrix", mat), ("grouped", grouped)):
            ms, _ = timed(torch, f)
            times[name].append(round(ms, 4))
    word = L * ctx.n * 8
    alg_bytes = (rows * inner + inner * cols) * 2 * word + rows * cols * 3 * word
    k = {}
    for name, ts in times.items():
        med = statistics.median(ts)
        k[name] = {"ms": ts, "median_ms": round(med, 4), "alg_TBps": round(alg_bytes / med / 1e9, 3),
                   "fraction_of_7.7TBps": round(alg_bytes / med / 1e9 / HBM_TBS, 3)}
    rec["contraction"] = {"rows": rows, "inner": inner, "cols": cols, "limbs": L, "algorithmic_bytes": alg_bytes,
                          "word_for_word_equal": bool(equal), "kernels": k,
                          "note": "matrix: one ckks_multiply_sum_matrix launch; grouped: t_p ckks_multiply_sum_grouped "
                                  "launches over B's columns gathered before the timing; random canonical residues"}
    print(json.dumps(rec["contraction"]), flush=True)
    os.makedirs(a.out_dir, exist_ok=True)
    path = os.path.join(a.out_dir, "matmul_blocked_1gpu.json")
    with open(path, "w") as fh:
        fh.write(json.dumps(rec, indent=1) + "\n")
    print(path)


if __name__ == "__main__":
    main()
