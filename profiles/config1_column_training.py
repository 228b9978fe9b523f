"""Config-1 training in the column layout with the Chebyshev sigmoid: 100 iterations of full-batch gradient descent
(column_epoch_gradient, apply_gradient, then the key holder's refresh of the packed weights and the weight broadcasts) on
the pulsar data, one GPU or several under torchrun, for each mini-batch size given.

    python profiles/config1_column_training.py [--iters 100] [--batch 2000 250] [--out-dir DIR]
    python -m torch.distributed.run --nproc_per_node G profiles/config1_column_training.py ...

Data: the 2000 x 8 rows of tests/golden/pulsar_stars.csv, standardised, the reference program's initial weights and
lr 0.1 (tests/golden/pulsar_plain_lr.json).  Sigmoid: lr.SIGMOID_CHEBYSHEV (degree 63 on [-48, 48]); N = 32768,
{60, 40 x 11, 60}, power-of-two Galois keys.  The iteration is parallel.sharded_train_columns with one iteration per call
(on one GPU: every unit on rank 0, the code path of lr.train_columns with phase marks); the M*C (mini-batch, feature)
units are split by parallel.column_units.

Rank 0 writes DIR/r06_config1_column_training_<G>gpu.json.  Per mini-batch size: the cost of the decrypted weights after
every iteration next to the reference program's cost history, max |dw| against plaintext Chebyshev LR (lr.plain_epoch,
same start) after every iteration, the final weights against the reference's, milliseconds per iteration (host clock
around one iteration and its refresh, ended by a device synchronise; slowest rank), the phases from CUDA events, the key
switches per rank counted from the partition, the levels used, bytes exchanged and peak memory per rank.  Then the
grouped product-sum of the prediction (ckks_multiply_sum_grouped) against the path it replaced (repeat of the
broadcasts, multiply, one add_many per mini-batch) at the pulsar shapes, alternated in this run, with their outputs
compared; and the GPU's name, power limit and maximum SM clock read in the same run."""
import argparse
import importlib
import json
import os
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
import config1_scaling  # noqa: E402  (CountingExchange with broadcast)
import matmul_scaling  # noqa: E402  (gpu_info)

PKG = "seal-fyp-logistic-regression_b200"
SCALE = 2.0 ** 40
CHAIN = [60] + [40] * 11 + [60]
PHASES = ("prediction", "polynomial", "gradient", "combine", "tail", "refresh")
HBM_TBS = 7.7          # HGX B200 data sheet, one GPU


def old_prediction_sum(ev, eng, cols, w_bcast, M):
    """the column prediction before ckks_multiply_sum_grouped: M copies of the broadcasts, M*C size-3 products, one
    add_many per mini-batch"""
    C = w_bcast.batch
    wb = eng.Ciphertext(w_bcast.ctx, w_bcast.data.repeat(M, 1, 1, 1), w_bcast.limbs, w_bcast.scale)
    prods = ev.multiply(cols, wb)
    z = [ev.add_many(prods[m * C:(m + 1) * C]) for m in range(M)]
    return eng.Ciphertext(cols.ctx, torch.cat([t.data for t in z], dim=0), prods.limbs, prods.scale)


def kernel_ab(eng, ctx, ev, M, C, reps):
    """old path vs ckks_multiply_sum_grouped at M mini-batches x C features, top level (12 limbs); the two alternate
    rep by rep, each timed with CUDA events; the inputs (M*C column ciphertexts, 0.4 / 0.8 GB at M = 8 / 16) exceed
    the 126 MB L2"""
    L = ctx.top_limbs
    cols, wb = ctx.empty(M * C, 2, L, scale=SCALE), ctx.empty(C, 2, L, scale=SCALE)
    for t in (cols, wb):
        for j in range(L):
            t.data[:, :, j].random_(0, ctx.primes[j])
    new = ev.multiply_sum_grouped(cols, wb, M)
    old = old_prediction_sum(ev, eng, cols, wb, M)
    same = bool(torch.equal(new.data[:, :, :L], old.data[:, :, :L]) and new.scale == old.scale)
    times = {"old": [], "new": []}
    fns = {"old": lambda: old_prediction_sum(ev, eng, cols, wb, M), "new": lambda: ev.multiply_sum_grouped(cols, wb, M)}
    for _ in range(reps):
        for k in ("old", "new"):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fns[k]()
            e1.record()
            torch.cuda.synchronize()
            times[k].append(e0.elapsed_time(e1))
    words = ctx.n * L
    nbytes = (M * C * 2 + C * 2 + M * 3) * words * 8          # read the columns and broadcasts once, write M size-3 sums
    res = {"M": M, "C": C, "limbs": L, "bit_identical": same, "algorithmic_bytes": nbytes, "reps": reps}
    for k in ("old", "new"):
        med = float(np.median(times[k]))
        res[k] = {"ms_median": med, "ms_all": times[k], "algorithmic_tb_per_s": nbytes / (med * 1e-3) / 1e12,
                  "share_of_hbm_7_7_tbs": nbytes / (med * 1e-3) / 1e12 / HBM_TBS}
    res["speedup_old_over_new"] = res["old"]["ms_median"] / res["new"]["ms_median"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--batch", type=int, nargs="+", default=[2000, 250], help="mini-batch sizes B (each divides 2000)")
    ap.add_argument("--kernel-reps", type=int, default=20)
    ap.add_argument("--out-dir", default=".", help="directory for the JSON (created if missing)")
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank = dist.get_rank() if world > 1 else 0

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
    gh = np.array(gold["cost_history"][:args.iters])

    ctx = eng.Context(15, params.coeff_modulus_create(15, CHAIN), device=local)
    ev, enc = eng.Evaluator(ctx), client.CKKSEncoder(ctx)
    kg = client.KeyGenerator(ctx, seed=91)                 # same keys and inputs on every rank
    keys = kg.keyset(steps=[s for i in range(13) for s in (1 << i, -(1 << i))])
    pk = kg.public_key()
    decr = client.Decryptor(ctx, kg.secret_key()) if rank == 0 else None
    events = []

    def mark(_name):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        events.append(e)

    runs = []
    for B in args.batch:
        lay = lr.ColumnLayout(R, C, B, ctx.n // 2)
        units = par.column_units(lay.M, C, rank, world)
        ids = sorted({m for m, _ in units})
        lo, hi = (ids[0], ids[-1] + 1) if ids else (0, 0)
        encr = client.Encryptor(ctx, pk, seed=92)
        cols = encr.encrypt(enc.encode(lay.columns(X), SCALE))
        labs = encr.encrypt(enc.encode(lay.labels(y), SCALE))
        wct = encr.encrypt(enc.encode(lay.weights(w0), SCALE))
        wb = encr.encrypt(enc.encode(lay.weight_broadcasts(w0, "chebyshev", sig), SCALE))
        cols_local = eng.Ciphertext(ctx, cols.data[lo * C:hi * C].clone(), cols.limbs, cols.scale)
        labs_local = eng.Ciphertext(ctx, labs.data[lo:hi].clone(), labs.limbs, labs.scale)
        del cols, labs
        key_holder = client.Encryptor(ctx, pk, seed=93) if rank == 0 else None
        ex = config1_scaling.CountingExchange(par)
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats(ctx.device)

        plain = w0.copy()
        costs, dw, times, phases = [], [], [], []
        for it in range(args.iters):
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            events.clear()
            mark("start")
            t0 = time.perf_counter()
            wct, wb = par.sharded_train_columns(ev, cols_local, labs_local, ids, units, wct, wb, rate, 1, lay, SCALE, keys,
                                                enc, key_holder, decr, rank, world, ex, sigmoid=sig, mark=mark)
            torch.cuda.synchronize()
            t = torch.tensor([(time.perf_counter() - t0) * 1e3], device=ctx.device)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)     # an iteration is done when its slowest rank is
            times.append(float(t.item()))
            phases.append([a.elapsed_time(b) for a, b in zip(events[:-1], events[1:])])
            plain = lr.plain_epoch(X, y, plain, rate, method="chebyshev", sigmoid=sig)
            if rank == 0:
                w = enc.decode(decr.decrypt(wct))[0, :C]
                costs.append(float(pulsar.cost_function(Xs, y, w)))
                dw.append(float(np.abs(w - plain).max()))
                print("B %d iteration %d: cost %.6f (reference %.6f), max |dw| vs plaintext %.2e, %.0f ms"
                      % (B, it, costs[-1], gh[it], dw[-1], times[-1]), flush=True)
        mine = [ex.sent // args.iters, ex.received // args.iters, torch.cuda.max_memory_allocated(ctx.device)]
        ph = np.median(np.array(phases), axis=0)
        if world > 1:
            allc = [torch.zeros(3, dtype=torch.int64, device=ctx.device) for _ in range(world)]
            dist.all_gather(allc, torch.tensor(mine, dtype=torch.int64, device=ctx.device))
            allp = [torch.zeros(len(PHASES), dtype=torch.float64, device=ctx.device) for _ in range(world)]
            dist.all_gather(allp, torch.tensor(ph, dtype=torch.float64, device=ctx.device))
            allc, allp = [c.tolist() for c in allc], [p.tolist() for p in allp]
        else:
            allc, allp = [mine], [ph.tolist()]
        if rank == 0:
            runs.append({
                "mini_batch": B, "mini_batches": lay.M, "units": lay.M * C,
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
                "ms_first_iteration": times[0],
                "ms_all": times,
                "phase_ms_median_per_rank": [dict(zip(PHASES, [float(v) for v in p])) for p in allp],
                "units_per_rank": [len(par.column_units(lay.M, C, q, world)) for q in range(world)],
                "key_switches_per_rank": [par.column_keyswitches(R, C, B, q, world, "chebyshev", sigmoid=sig)
                                          for q in range(world)],
                "key_switches_one_gpu": par.column_keyswitches(R, C, B, 0, 1, "chebyshev", sigmoid=sig),
                "bytes_sent_per_rank_per_iteration": [int(c[0]) for c in allc],
                "bytes_received_per_rank_per_iteration": [int(c[1]) for c in allc],
                "peak_torch_allocated_bytes_per_rank": [int(c[2]) for c in allc],
            })
        del cols_local, labs_local

    kernel = [kernel_ab(eng, ctx, ev, M, C, args.kernel_reps) for M in (8, 16)] if rank == 0 else None
    if rank == 0:
        res = {
            "workload": "config 1 in the column layout: full-batch gradient descent with the Chebyshev sigmoid (degree %d "
                        "on [-%g, %g]) on pulsar_stars.csv 2000 x 8 standardised, the reference program's initial weights, "
                        "lr %g, %d iterations with refresh; N=32768 {60,40x11,60}, power-of-two Galois keys, %d GPU(s)"
                        % (sig.degree, sig.bound, sig.bound, rate, args.iters, world),
            "gpus": world, "gpu": matmul_scaling.gpu_info(local), "iterations": args.iters,
            "runs": runs,
            "timing": "host clock around one sharded_train_columns iteration (prediction, polynomial, gradient, combine, "
                      "learning-rate tail, rank 0's decrypt / decode / encode / encrypt of the weights and broadcasts, "
                      "their broadcast), ended by a device synchronise; slowest rank",
            "phases": "CUDA events at the end of each phase on each rank's stream, median over the iterations; a phase "
                      "that waits for another rank (combine, refresh) includes the wait",
            "levels": {"data_primes": len(CHAIN) - 1, "rescales_per_iteration": lr.column_rescales("chebyshev", sigmoid=sig),
                       "prediction": 1, "polynomial": wl.chebyshev_depth(sig.degree), "dot_product": 1, "mask": 1,
                       "learning_rate": 1},
            "relinearisations_polynomial_per_mini_batch": wl.chebyshev_keyswitches(sig.degree),
            "memory": "peak of torch's allocator over the iterations of one mini-batch size (keys, own column and label "
                      "ciphertexts, weights, broadcasts and the iteration's intermediates)",
            "prediction_kernel_ab": kernel,
            "prediction_kernel_note": "ckks_multiply_sum_grouped ('new') against repeat + multiply + add_many per "
                                      "mini-batch ('old') at N=32768, 12 limbs, alternated rep by rep; algorithmic bytes "
                                      "= columns and broadcasts read once + the M size-3 sums written, over the %.1f TB/s "
                                      "HBM figure of the B200 data sheet" % HBM_TBS,
        }
        os.makedirs(args.out_dir, exist_ok=True)
        path = os.path.join(args.out_dir, "r06_config1_column_training_%dgpu.json" % world)
        with open(path, "w") as fh:
            json.dump(res, fh, indent=1)
        print(json.dumps({"gpu": res["gpu"], "runs": [{k: r[k] for k in (
            "mini_batch", "max_abs_cost_diff_vs_reference", "max_abs_dw_vs_plaintext_chebyshev_lr_max",
            "max_abs_final_weights_diff_vs_reference", "ms_per_iteration_median", "phase_ms_median_per_rank")} for r in runs],
            "kernel": [{"M": k["M"], "same": k["bit_identical"], "old_ms": k["old"]["ms_median"],
                        "new_ms": k["new"]["ms_median"]} for k in kernel]}), flush=True)
        print("wrote", path, flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
