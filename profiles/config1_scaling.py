"""Strong scaling of one config-1 training iteration (BASELINE config 1: the reference's update_weights, row layout,
Horner degree 3, lr 0.1; N = 32768, {60, 40 x 8, 60}, power-of-two Galois keys; the set-up of bench.py: config1_pulsar)
sharded with parallel.sharded_update_weights over the GPUs of one node.

    python -m torch.distributed.run --nproc_per_node G profiles/config1_scaling.py [--reps 3] [--warmup 1]
        [--rows R] [--out-dir DIR]

Without --rows the data are the 2000 x 8 rows of tests/golden/pulsar_stars.csv, standardised, with the reference
program's initial weights (tests/golden/pulsar_plain_lr.json).  --rows R runs R synthetic rows of 8 standard-normal
features instead (2R <= N/2: R <= 8192), to show how the gradient chains of R - 1 dependent rotations grow.

Every rank encrypts the whole data set from the same seeds, in fixed chunks of rows, and keeps only its own row and
feature blocks, so that rank 0 can rebuild the unsharded inputs afterwards and check bit-identity.  Rank 0 writes
DIR/r04_config1_scaling_<G>gpu.json (with --rows: ..._<G>gpu_rows<R>.json): milliseconds per iteration (host clock
around one iteration ended by a device synchronise on every rank, slowest rank per repetition), the time of each phase
on each rank from CUDA events, key switches per rank counted from the partition, bytes sent and received per rank, peak
device memory per rank, bit-identity with the unsharded lr.update_weights (rank 0 also times it once), max |dw| against
plaintext LR with the same polynomial, and the GPU's name, power limit and maximum SM clock read in the same run."""
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
import matmul_scaling  # noqa: E402  (gpu_info, CountingExchange)

PKG = "seal-fyp-logistic-regression_b200"
SCALE, LR, DEGREE, CHUNK = 2.0 ** 40, 0.1, 3, 500
CHAIN = [60] + [40] * 8 + [60]
PHASES = ("prediction", "combine_prediction", "polynomial_broadcast", "gradient", "combine_gradient", "tail")


class CountingExchange(matmul_scaling.CountingExchange):
    """the byte-counting exchange of matmul_scaling.py plus the broadcast of the config-1 iteration"""

    def broadcast(self, t, src=0):
        nb = t.numel() * t.element_size()
        if self.world > 1:
            if self.rank == src:
                self.sent += nb * (self.world - 1)
            else:
                self.received += nb
        return self.inner.broadcast(t, src)


def load_data(rows):
    pulsar = importlib.import_module(PKG + ".pulsar")
    if rows:
        rng = np.random.default_rng(rows)
        X = rng.normal(0, 1, (rows, 8))
        return X, (rng.uniform(0, 1, rows) > 0.5).astype(np.float64), rng.uniform(-1, 1, 8), "synthetic %d x 8" % rows
    with open(os.path.join(ROOT, "tests", "golden", "pulsar_plain_lr.json")) as fh:
        w0 = np.array(json.load(fh)["initial_weights"])
    X, y = pulsar.load_csv()
    return (pulsar.standard_scaler(X).astype(np.float64), y.astype(np.float64), w0,
            "pulsar_stars.csv (2000 x 8, standardised, the reference program's initial weights)")


def encrypt_inputs(ctx, enc, encr, lay, X, y, w0, row_block=None, feature_block=None):
    """rows (in chunks of CHUNK), columns, labels, weights, always in this order with one encryptor; with blocks given
    only those rows / columns are kept"""
    eng = importlib.import_module(PKG + ".engine")
    R = X.shape[0]
    row_block = range(R) if row_block is None else row_block
    packed = lay.rows(X)
    kept = []
    for s in range(0, R, CHUNK):
        ct = encr.encrypt(enc.encode(packed[s:s + CHUNK], SCALE))
        lo, hi = max(s, row_block.start), min(s + CHUNK, row_block.stop)
        if lo < hi:
            kept.append(ct.data[lo - s:hi - s].clone())
        limbs, scale, shape = ct.limbs, ct.scale, ct.data.shape
        del ct
    data = torch.cat(kept) if kept else torch.empty((0,) + tuple(shape[1:]), dtype=torch.int64, device=ctx.device)
    rows = eng.Ciphertext(ctx, data, limbs, scale)
    cols = encr.encrypt(enc.encode(lay.columns(X), SCALE))
    if feature_block is not None:
        cols = eng.Ciphertext(ctx, cols.data[feature_block.start:feature_block.stop].clone(), cols.limbs, cols.scale)
    labs = encr.encrypt(enc.encode(lay.labels(y), SCALE))
    wct = encr.encrypt(enc.encode(lay.weights(w0), SCALE))
    return rows, cols, labs, wct


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--rows", type=int, default=0, help="synthetic rows instead of the pulsar data (8 .. 8192)")
    ap.add_argument("--out-dir", default=".", help="directory for the JSON (created if missing)")
    args = ap.parse_args()
    if args.rows and not 8 <= args.rows <= 8192:
        ap.error("--rows must lie in [8, 8192] (2R <= N/2)")
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()

    eng = importlib.import_module(PKG).load_engine()
    lr, par = importlib.import_module(PKG + ".lr"), importlib.import_module(PKG + ".parallel")
    client, params = importlib.import_module(PKG + ".client"), importlib.import_module(PKG + ".params")
    ctx = eng.Context(15, params.coeff_modulus_create(15, CHAIN), device=local)
    ev = eng.Evaluator(ctx)
    enc = client.CKKSEncoder(ctx)
    kg = client.KeyGenerator(ctx, seed=71)                 # same keys and inputs on every rank
    keys = kg.keyset(steps=[s for i in range(13) for s in (1 << i, -(1 << i))])
    pk = kg.public_key()                                   # drawn once: every Encryptor below must use the same key
    X, y, w0, what = load_data(args.rows)
    R, C = X.shape
    lay = lr.RowLayout(R, C, ctx.n // 2)
    rb, fb = par.config1_shards(R, C, rank, world)
    rows, cols, labs, wct = encrypt_inputs(ctx, enc, client.Encryptor(ctx, pk, seed=72), lay, X, y, w0, rb, fb)
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats(ctx.device)

    ex = CountingExchange(par)
    events = []

    def mark(_name):
        ev_ = torch.cuda.Event(enable_timing=True)
        ev_.record()
        events.append(ev_)

    def run():
        # the key holder's encryptor starts from the same seed every iteration: every repetition computes the same
        # ciphertext, the one the unsharded check below reproduces
        encr = client.Encryptor(ctx, pk, seed=73) if rank == 0 else None
        return par.sharded_update_weights(ev, rows, list(rb), cols, list(fb), labs, wct, LR, R, C, SCALE, keys, enc, encr,
                                          rank, world, ex, degree=DEGREE, mark=mark)

    for _ in range(args.warmup):
        out = run()
    torch.cuda.synchronize()
    ex.sent = ex.received = 0
    times, phases = [], []
    for _ in range(args.reps):
        dist.barrier()
        torch.cuda.synchronize()
        events.clear()
        mark("start")
        t0 = time.perf_counter()
        out = run()
        torch.cuda.synchronize()
        t = torch.tensor([(time.perf_counter() - t0) * 1e3], device=ctx.device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)            # an iteration is done when its slowest rank is
        times.append(float(t.item()))
        phases.append([a.elapsed_time(b) for a, b in zip(events[:-1], events[1:])])
    free, total = torch.cuda.mem_get_info(ctx.device)
    mine = [ex.sent // args.reps, ex.received // args.reps, torch.cuda.max_memory_allocated(ctx.device), total - free]
    allc = [torch.zeros(4, dtype=torch.int64, device=ctx.device) for _ in range(world)]
    dist.all_gather(allc, torch.tensor(mine, dtype=torch.int64, device=ctx.device))
    ph = torch.tensor(np.median(np.array(phases), axis=0), dtype=torch.float64, device=ctx.device)
    allp = [torch.zeros_like(ph) for _ in range(world)]
    dist.all_gather(allp, ph)

    if rank == 0:
        del rows, cols
        torch.cuda.empty_cache()
        full = encrypt_inputs(ctx, enc, client.Encryptor(ctx, pk, seed=72), lay, X, y, w0)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        want = lr.update_weights(ev, *full, LR, SCALE, keys, enc, client.Encryptor(ctx, pk, seed=73),
                                 degree=DEGREE)
        torch.cuda.synchronize()
        ms_unsharded = (time.perf_counter() - t0) * 1e3
        same = bool(out.limbs == want.limbs and out.scale == want.scale and
                    torch.equal(out.data[:, :, :out.limbs], want.data[:, :, :want.limbs]))
        dec = client.Decryptor(ctx, kg.secret_key())
        plain = lr.plain_epoch(X, y, w0, LR, DEGREE)
        err = float(np.abs(enc.decode(dec.decrypt(out))[0, :C] - plain).max())
        err_unsharded = float(np.abs(enc.decode(dec.decrypt(want))[0, :C] - plain).max())
        per_rank = [[float(v) for v in p.tolist()] for p in allp]
        med = float(np.median(times))
        res = {
            "workload": "config 1: update_weights on %s, row layout, Horner degree 3, lr 0.1, N=32768 {60,40x8,60}, "
                        "power-of-two Galois keys, rows and features sharded over %d GPU(s)" % (what, world),
            "gpus": world, "gpu": matmul_scaling.gpu_info(local), "rows": R, "features": C,
            "ms_per_iteration": med, "ms_min": min(times), "ms_max": max(times), "ms_all": times,
            "timing": "host clock around one iteration ended by a device synchronise on every rank, slowest rank, "
                      "%d repetitions after %d warm-up" % (args.reps, args.warmup),
            "iterations_per_s": 1e3 / med,
            "phase_ms_per_rank": [dict(zip(PHASES, p)) for p in per_rank],
            "phase_ms_sum_per_rank": [sum(p) for p in per_rank],
            "phases": "CUDA events on each rank's stream at the end of each phase, median over the repetitions; a phase "
                      "that waits for another rank (combine, broadcast) includes the wait",
            "ms_unsharded_one_gpu": ms_unsharded,
            "rows_per_rank": [len(par.config1_shards(R, C, q, world)[0]) for q in range(world)],
            "features_per_rank": [len(par.config1_shards(R, C, q, world)[1]) for q in range(world)],
            "key_switches_per_rank": [par.config1_keyswitches(R, C, q, world, DEGREE) for q in range(world)],
            "key_switches_one_gpu": par.config1_keyswitches(R, C, 0, 1, DEGREE),
            "bytes_sent_per_rank": [int(c[0]) for c in allc], "bytes_received_per_rank": [int(c[1]) for c in allc],
            "peak_torch_allocated_bytes_per_rank": [int(c[2]) for c in allc],
            "device_memory_used_bytes_per_rank": [int(c[3]) for c in allc],
            "memory": "peak of torch's allocator over the timed iterations (keys, own row / feature ciphertexts, labels, "
                      "weights and the iteration's intermediates); device_memory_used = total - free after them (also "
                      "the engine's workspace and the allocator's cache)",
            "bit_identical": same,
            "max_abs_err_vs_plaintext_polynomial_lr": err,
            "max_abs_err_unsharded_vs_plaintext_polynomial_lr": err_unsharded,
        }
        os.makedirs(args.out_dir, exist_ok=True)
        name = "r04_config1_scaling_%dgpu%s.json" % (world, "_rows%d" % R if args.rows else "")
        path = os.path.join(args.out_dir, name)
        with open(path, "w") as fh:
            json.dump(res, fh, indent=1)
        print(json.dumps({k: res[k] for k in ("gpus", "rows", "ms_per_iteration", "ms_min", "ms_max", "ms_unsharded_one_gpu",
                                              "phase_ms_sum_per_rank", "bit_identical",
                                              "max_abs_err_vs_plaintext_polynomial_lr", "key_switches_per_rank")}),
              flush=True)
        print("wrote", path, flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
