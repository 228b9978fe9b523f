"""Encrypted config-1 training with the Chebyshev sigmoid: 100 iterations of the reference's train_cipher (update_weights,
then the key holder decrypts, re-encodes and re-encrypts the weights) on the pulsar data, one GPU.

    python profiles/config1_chebyshev_training.py [--iters 100] [--out-dir DIR]

Data: the 2000 x 8 rows of tests/golden/pulsar_stars.csv, standardised, the reference program's initial weights and
lr 0.1 (tests/golden/pulsar_plain_lr.json).  Sigmoid: lr.SIGMOID_CHEBYSHEV (degree 63 on [-48, 48]), evaluated by
workloads.chebyshev_cipher; N = 32768, {60, 40 x 12, 60}, power-of-two Galois keys.  The iteration is
parallel.sharded_update_weights on one rank (the code path of lr.update_weights with phase marks).

Writes DIR/r05_config1_chebyshev_training_1gpu.json: the cost of the decrypted weights after every iteration next to the
reference program's printed cost history, max |dw| against plaintext Chebyshev LR (lr.plain_epoch, same start) after
every iteration, the final weights against the reference's, milliseconds per iteration (host clock around the iteration
and its refresh, ended by a device synchronise) and per phase (CUDA events), the levels used, and the GPU's name, power
limit and maximum SM clock read in the same run."""
import argparse
import importlib
import json
import os
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
import matmul_scaling  # noqa: E402  (gpu_info)

PKG = "seal-fyp-logistic-regression_b200"
SCALE = 2.0 ** 40
CHAIN = [60] + [40] * 12 + [60]
PHASES = ("prediction", "combine_prediction", "polynomial", "gradient", "combine_gradient", "tail", "refresh")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--out-dir", default=".", help="directory for the JSON (created if missing)")
    args = ap.parse_args()

    eng = importlib.import_module(PKG).load_engine()
    lr, par, wl = (importlib.import_module(PKG + m) for m in (".lr", ".parallel", ".workloads"))
    client, params, pulsar = (importlib.import_module(PKG + m) for m in (".client", ".params", ".pulsar"))
    with open(os.path.join(ROOT, "tests", "golden", "pulsar_plain_lr.json")) as fh:
        gold = json.load(fh)
    X, y = pulsar.load_csv()
    Xs = pulsar.standard_scaler(X)
    X, y = Xs.astype(np.float64), y.astype(np.float64)
    w0, rate = np.array(gold["initial_weights"]), float(gold["learning_rate"])
    R, C = X.shape
    sig = lr.SIGMOID_CHEBYSHEV

    ctx = eng.Context(15, params.coeff_modulus_create(15, CHAIN))
    ev, enc = eng.Evaluator(ctx), client.CKKSEncoder(ctx)
    kg = client.KeyGenerator(ctx, seed=81)
    keys = kg.keyset(steps=[s for i in range(13) for s in (1 << i, -(1 << i))])
    encr, decr = client.Encryptor(ctx, kg.public_key(), seed=82), client.Decryptor(ctx, kg.secret_key())
    lay = lr.RowLayout(R, C, ctx.n // 2)
    rows = encr.encrypt(enc.encode(lay.rows(X), SCALE))
    cols = encr.encrypt(enc.encode(lay.columns(X), SCALE))
    labs = encr.encrypt(enc.encode(lay.labels(y), SCALE))
    wct = encr.encrypt(enc.encode(lay.weights(w0), SCALE))
    ex = par.TorchExchange()
    events = []

    def mark(_name):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        events.append(e)

    plain = w0.copy()
    costs, dw, times, phases = [], [], [], []
    for it in range(args.iters):
        torch.cuda.synchronize()
        events.clear()
        mark("start")
        t0 = time.perf_counter()
        out = par.sharded_update_weights(ev, rows, list(range(R)), cols, list(range(C)), labs, wct, rate, R, C, SCALE, keys,
                                         enc, None, 0, 1, ex, method="chebyshev", mark=mark, sigmoid=sig)
        limbs_after = out.limbs
        w = enc.decode(decr.decrypt(out))[0, :C]
        wct = encr.encrypt(enc.encode(lay.weights(w), SCALE))
        mark("refresh")
        torch.cuda.synchronize()
        times.append((time.perf_counter() - t0) * 1e3)
        phases.append([a.elapsed_time(b) for a, b in zip(events[:-1], events[1:])])
        plain = lr.plain_epoch(X, y, plain, rate, method="chebyshev", sigmoid=sig)
        costs.append(float(pulsar.cost_function(Xs, y, w)))
        dw.append(float(np.abs(w - plain).max()))
        print("iteration %d: cost %.6f (reference %.6f), max |dw| vs plaintext %.2e, %.0f ms"
              % (it, costs[-1], gold["cost_history"][it], dw[-1], times[-1]), flush=True)

    gh = np.array(gold["cost_history"][:args.iters])
    res = {
        "workload": "config 1 train_cipher with the Chebyshev sigmoid (degree %d on [-%g, %g]): pulsar_stars.csv 2000 x 8 "
                    "standardised, the reference program's initial weights, lr %g, %d iterations with refresh; N=32768 "
                    "{60,40x12,60}, power-of-two Galois keys, one GPU" % (sig.degree, sig.bound, sig.bound, rate, args.iters),
        "gpu": matmul_scaling.gpu_info(0),
        "iterations": args.iters,
        "cost_encrypted": costs,
        "cost_reference": [float(v) for v in gh],
        "max_abs_cost_diff_vs_reference": float(np.abs(np.array(costs) - gh).max()),
        "max_abs_dw_vs_plaintext_chebyshev_lr": dw,
        "max_abs_dw_vs_plaintext_chebyshev_lr_max": max(dw),
        "final_weights_encrypted": [float(v) for v in w],
        "final_weights_reference": gold["final_weights"],
        "max_abs_final_weights_diff_vs_reference": float(np.abs(w - np.array(gold["final_weights"])).max())
        if args.iters == gold["iterations"] else None,
        "ms_per_iteration_median": float(np.median(times)),
        "ms_per_iteration_mean": float(np.mean(times)),
        "ms_first_iteration": times[0],
        "ms_all": times,
        "timing": "host clock around update_weights + decrypt / decode / encode / encrypt of the weights, ended by a "
                  "device synchronise",
        "phase_ms_median": dict(zip(PHASES, [float(v) for v in np.median(np.array(phases), axis=0)])),
        "phases": "CUDA events at the end of each phase of parallel.sharded_update_weights (one rank; 'polynomial' is the "
                  "rescale, chebyshev_cipher and the label subtraction), then the refresh; median over the iterations",
        "levels": {"data_primes": len(CHAIN) - 1, "polynomial": wl.chebyshev_depth(sig.degree),
                   "prediction": 2, "gradient_and_tail": 3, "limbs_left_after_iteration": limbs_after},
        "relinearisations_polynomial": wl.chebyshev_keyswitches(sig.degree),
        "key_switches_per_iteration": par.config1_keyswitches(R, C, 0, 1, method="chebyshev", sigmoid=sig),
    }
    os.makedirs(args.out_dir, exist_ok=True)
    path = os.path.join(args.out_dir, "r05_config1_chebyshev_training_1gpu.json")
    with open(path, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({k: res[k] for k in ("gpu", "max_abs_cost_diff_vs_reference", "max_abs_dw_vs_plaintext_chebyshev_lr_max",
                                          "max_abs_final_weights_diff_vs_reference", "ms_per_iteration_median",
                                          "phase_ms_median")}), flush=True)
    print("wrote", path, flush=True)


if __name__ == "__main__":
    main()
