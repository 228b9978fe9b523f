#!/usr/bin/env python
"""bench.py -- encrypted logistic-regression training throughput on B200 (BASELINE.json metric
"CKKS LR train epochs/s; rotate/relin keyswitch ops/s at N=2^14,2^15").

Workload (BASELINE.json configs[4], SURVEY.md 8(d) config 5): synthetic 8 features x 32768 samples,
N = 32768, coeff_modulus {60, 40 x 8, 60}, scale 2^40, tree-method degree-7 sigmoid, column layout with
mini-batches of 8192 samples.  One step = one epoch: for every mini-batch  z = sum_j multiply(col_j, w_j);
relinearize; rescale; Tree_cipher(z); sub labels; per feature cipher_dot_product(col_j, pred - y, 8192)
(1 relinearize + 8192 Galois key switches at L = 3) and the one-hot mask; add_many; rescale -- then the
partial gradient ciphertexts of all GPUs are all-gathered (NCCL) and combined with the mod-q add kernel,
and the weight update (multiply_plain lr/R, rescale, sub, negate) is applied.

Scaling (--scaling, default "strong" = what BASELINE config 5 describes: "gradient ciphertexts sharded over
1/2/4/8 B200"): ONE 8 x 32768 problem; its 32 (mini-batch, feature) gradient chains are split over the N
GPUs (4 chains per GPU at N = 8), every GPU evaluates the prediction of the mini-batches it touches.
"weak": every GPU holds its own 8 x 32768 shard (N problems); reported as the extra key `weak_scaling`
when N > 1.  At N = 1 the two coincide.

  python bench.py --gpus N --steps K --warmup W      (N > 1 under torch.distributed.run)
  python bench.py ... --dump-outputs DIR             also write the last timed epoch's outputs to DIR/*.npy
  python bench.py --impl reference ...               CPU arm: the SEAL-3.4.5-equivalent oracle
                                                     (SEAL itself is not installable here) on the
                                                     host cores, bounded sample, same metric

Prints ONE JSON line on rank 0.
"""
import argparse
import importlib
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
PKG = "seal-fyp-logistic-regression_b200"

LOG_N = 15
BITS = [60] + [40] * 8 + [60]
SCALE = 2.0 ** 40
C_FEAT = 8
R_PER_GPU = 32768            # samples of the problem (strong) / of every GPU's shard (weak)
B_MINI = 8192
DEGREE = 7
LR = 0.1
METRIC = "ckks_lr_train_epochs_per_s"
UNIT = "epochs/s"


def ks_bytes(L, n, relin=False):
    """algorithmic bytes of one key switch (SURVEY.md 8(d)): rotate (2L^2+6L)*8N, relin (2L^2+7L)*8N"""
    return (2 * L * L + (7 if relin else 6) * L) * 8 * n


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------ clocks
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.samples, self.proc = [], None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(index), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.samples:
            if ts < t0 or ts > t1:
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except Exception:
                continue
            for name, val in zip(names, f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------ data
def synthetic_shard(seed):
    rng = np.random.default_rng(seed)
    X = rng.normal(0.0, 1.0, (R_PER_GPU, C_FEAT))
    w_true = rng.uniform(-1, 1, C_FEAT)
    y = (1.0 / (1.0 + np.exp(-X @ w_true)) > rng.uniform(0, 1, R_PER_GPU)).astype(np.float64)
    return X, y


def epoch_op_counts():
    """evaluator ops of one epoch on one GPU, by (op, limbs): used to scale the CPU sample"""
    M, C, B = R_PER_GPU // B_MINI, C_FEAT, B_MINI
    top = len(BITS) - 1
    ops = []
    ops += [("multiply", top, M * C), ("add3", top, M * (C - 1)), ("relinearize", top, M), ("rescale", top, M)]
    # tree degree 7: x at L8; x^2 L8->7, x^3 / x^4 at L7->6, x^5..x^7 at L6->5
    for lvl, cnt in ((top - 1, 1), (top - 2, 2), (top - 3, 3)):
        ops += [("multiply", lvl, M * cnt), ("relinearize", lvl, M * cnt), ("rescale", lvl, M * cnt)]
    ops += [("multiply_plain", top - 3, M * 7), ("rescale", top - 3, M * 7), ("add", top - 5, M * 8)]
    Lp = top - 5                                   # level of the prediction (4)
    ops += [("multiply", Lp, M * C), ("relinearize", Lp, M * C), ("rescale", Lp, M * C)]
    ops += [("rotate", Lp - 1, M * C * B), ("add", Lp - 1, M * C * B)]
    ops += [("multiply_plain", Lp - 1, M * C), ("add", Lp - 1, M * C), ("rescale", Lp - 1, 1)]
    return ops


# ------------------------------------------------------------------------------------ CPU arm
def cpu_reference(budget_s=20.0, threads=None, single_thread_s=4.0):
    """Time the CPU oracle (SEAL-3.4.5-equivalent restatement, gcc -O3 -march=native) on a bounded sample of the
    epoch.  The sample is a contiguous piece of the real op sequence, not isolated ops: every host thread runs ONE
    (mini-batch, feature) gradient unit of update_weights from its start -- cipher_dot_product = multiply,
    relinearize, rescale (L 4 -> 3), rotate_vector(-8192), add, then the dependent loop `rotate_vector(dup, 1);
    add_inplace(acc, dup)` (helper.h:416-476) -- and stops the loop after n of its 8191 iterations (n set by the
    time budget; n = 8191 would be the complete unit, ~2 min per thread).  The epoch time is then MODELLED:
    the loop iterations carry 99.97 % of an epoch's key switches, so
        epoch_s = (iterations per epoch / threads) x measured seconds per iteration with all threads busy
                  + the remaining ops (each timed once) x their counts / threads.
    SEAL itself is single-threaded; `single_thread` reports the same loop on one thread with the others idle."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import pyoracle as po
    threads = threads or (os.cpu_count() or 1)
    primes = po.coeff_modulus_create(LOG_N, BITS)
    orc = po.Oracle(LOG_N, primes)
    sk = orc.gen_secret(1)
    rlk = orc.gen_relin_key(2, sk)
    g1, gB = orc.galois_elt(1), orc.galois_elt(-B_MINI)
    gk1, gkB = orc.gen_galois_key(3, sk, g1), orc.gen_galois_key(4, sk, gB)
    rng = np.random.default_rng(0)
    n = 1 << LOG_N

    def rand_ct(S, L):
        return np.stack([rng.integers(0, p, size=(S, n), dtype=np.uint64) for p in primes[:L]], axis=1)

    L3 = len(BITS) - 1 - 6
    Lp = L3 + 1

    def unit(col, pl, iters, out):
        """one (mini-batch, feature) unit, truncated after `iters` loop iterations"""
        t0 = time.perf_counter()
        mult = orc.rescale(orc.relinearize(orc.multiply(col, pl), rlk))
        dup = orc.add(mult, orc.apply_galois(mult, gB, gkB))
        t1 = time.perf_counter()
        for _ in range(iters):
            dup = orc.apply_galois(dup, g1, gk1)
            mult = orc.add(mult, dup)
        out.append((t1 - t0, time.perf_counter() - t1))
        return mult

    # single thread, others idle (SEAL's own execution model)
    c0, p0 = rand_ct(2, Lp), rand_ct(2, Lp)
    probe = []
    unit(c0, p0, 3, probe)
    t_it = probe[0][1] / 3
    st = []
    it1 = max(4, int(single_thread_s / t_it))
    unit(c0, p0, it1, st)
    t_single = st[0][1] / it1
    # all threads
    iters = max(4, int(budget_s / (t_it * 1.8)))           # contention makes an iteration ~1.5-2x slower
    data = [(rand_ct(2, Lp), rand_ct(2, Lp)) for _ in range(threads)]
    outs = [[] for _ in range(threads)]
    t0 = time.perf_counter()
    with ThreadPoolExecutor(threads) as ex:
        list(ex.map(lambda k: unit(data[k][0], data[k][1], iters, outs[k]), range(threads)))
    wall = time.perf_counter() - t0
    t_head = float(np.mean([o[0][0] for o in outs]))        # multiply + relinearize + rescale + rotate(-B) + add, per unit
    t_loop = float(np.mean([o[0][1] for o in outs])) / iters  # seconds per (rotate 1 + add) per thread, all threads busy

    cache = {}

    def op_time(op, L):
        key = (op, L)
        if key not in cache:
            a2, b2, a3, pt = rand_ct(2, L), rand_ct(2, L), rand_ct(3, L), rand_ct(1, L)[0]
            fns = {
                "multiply": lambda: orc.multiply(a2, b2), "add3": lambda: orc.add(a3, a3), "add": lambda: orc.add(a2, b2),
                "relinearize": lambda: orc.relinearize(a3, rlk), "rescale": lambda: orc.rescale(a2),
                "multiply_plain": lambda: orc.multiply_plain(a2, pt),
            }
            t = time.perf_counter()
            fns[op]()
            cache[key] = time.perf_counter() - t
        return cache[key]

    M, C, B = R_PER_GPU // B_MINI, C_FEAT, B_MINI
    units = M * C
    loop_s = units * (B - 1) * t_loop / threads
    head_s = units * t_head / threads
    other_s = 0.0
    for op, L, cnt in epoch_op_counts():
        if (op in ("rotate", "add") and L == L3 and cnt > 1000) or (L == Lp and op in ("multiply", "relinearize", "rescale") and cnt == units):
            continue                                        # inside the measured unit
        other_s += cnt * op_time(op, L) / threads
    total = loop_s + head_s + other_s
    total_single = units * (B - 1) * t_single + (head_s + other_s) * threads
    return {
        "value": 1.0 / total, "unit": UNIT, "cores": threads, "kind": "port", "modelled": True,
        "sample": "%d threads x one (mini-batch, feature) gradient unit each (multiply, relinearize, rescale, rotate(-%d), add, "
                  "then %d of its %d dependent rotate(1)+add iterations), N=32768, L=%d, measured in %.1f s wall; "
                  "epoch time MODELLED = %d units x %d iterations x %.2f ms / %d threads + head %.2f s + other ops %.2f s = %.0f s" % (
                      threads, B, iters, B - 1, L3, wall, units, B - 1, 1e3 * t_loop, threads, head_s, other_s, total),
        "measured_wall_s": wall, "loop_iterations_measured_per_thread": iters,
        "rotate_add_ms_per_thread_all_threads_busy": 1e3 * t_loop,
        "single_thread": {"value": 1.0 / total_single, "unit": UNIT, "rotate_add_ms": 1e3 * t_single,
                          "iterations_measured": it1, "epoch_s_modelled": total_single},
        "oracle_build": "gcc -O3 -march=native (oracle/Makefile)",
    }


def run_reference(args):
    """--impl reference: the CPU arm alone.  A CPU epoch takes minutes (see `sample`), so the run cannot execute
    K real epochs inside the driver's window: ONE bounded sample is measured (all host threads, ~40 s) and every
    one of the K 'steps' is that sample scaled to an epoch -- `modelled: true`, `measured_wall_s` says what ran."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = max(1, args.steps)
    cb = cpu_reference(budget_s=max(args.cpu_budget, 30.0), single_thread_s=6.0)
    value = cb["value"]
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": args.warmup, "ms_per_step": 1e3 / value, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": workload_config(args.gpus, "strong"),
        "cpu_baseline": cb, "modelled": True,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "SEAL is not installable here (no source in the reference, no network); this arm times the "
                "SEAL-3.4.5-equivalent CPU oracle (kind: port) on ONE bounded sample of the same workload with all host "
                "threads and scales it to an epoch: value and ms_per_step are MODELLED from measured_wall_s of real work, "
                "they are not K measured epochs (one CPU epoch takes minutes).  The CPU holds the whole problem, so the "
                "value does not depend on --gpus.",
    }
    print(json.dumps(line))


def workload_config(n_gpus, scaling="strong"):
    per = "problem" if scaling == "strong" else "GPU"
    return {
        "workload": "encrypted LR training epoch, synthetic %d features x %d samples per %s, N=32768, "
                    "coeff_modulus {60,40x8,60}, scale 2^40, tree degree-%d sigmoid, column layout, "
                    "mini-batches of %d" % (C_FEAT, R_PER_GPU, per, DEGREE, B_MINI),
        "poly_modulus_degree": 1 << LOG_N, "coeff_modulus_bits": BITS, "features": C_FEAT,
        "samples": R_PER_GPU if scaling == "strong" else R_PER_GPU * n_gpus, "mini_batch": B_MINI,
        "sigmoid": "tree degree %d" % DEGREE,
        "parallelism": ("the 32 (mini-batch, feature) gradient chains of ONE problem split over %d GPU(s)" if scaling == "strong"
                        else "one 8 x 32768 shard per GPU, %d GPU(s)") % n_gpus + ", all-gather + mod-q add of the partial gradient ciphertexts",
        "l2_policy": "inputs exceed L2 (151 MB of column ciphertexts + 2 x 47 MB keys + 255 MB workspace per step at 1 GPU)",
    }


def dump_outputs(path, grad, neww, weights):
    """What a caller of the timed epoch receives, as float64 .npy files (3 MB in all): the gradient and updated weight
    ciphertexts and the decrypted updated weights.  A ciphertext's RNS residues [batch][size][limbs][N] reach 2^60, more
    than float64 holds exactly, so each is stored as two exact halves: <name>_hi = residue >> 30, <name>_lo = residue mod
    2^30.  Every epoch encrypts the sigmoid's constant term afresh (Tree_cipher) from the seeded encryptor's stream, so
    the arrays depend on how many epochs ran before the last one (--warmup, --steps); the public key is drawn after the
    doubling mode's Galois keys, so they also depend on --no-fast.  Runs with the same arguments write the same arrays."""
    os.makedirs(path, exist_ok=True)
    arrays = {"weights": np.asarray(weights, dtype=np.float64)}
    for name, ct in (("gradient_ct", grad), ("weights_ct", neww)):
        words = ct.numpy()
        arrays[name + "_hi"] = (words >> np.uint64(30)).astype(np.float64)
        arrays[name + "_lo"] = (words & np.uint64((1 << 30) - 1)).astype(np.float64)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


# ------------------------------------------------------------------------------------ GPU arm
def strong_units(rank, world):
    """(mini-batch, feature) gradient units of `rank` when ONE problem is split over `world` GPUs: a contiguous block
    of the M*C = 32 units in (m, j) order -- whole mini-batches per GPU up to 4 GPUs, half a mini-batch's features at 8"""
    total = (R_PER_GPU // B_MINI) * C_FEAT
    if total % world:
        raise SystemExit("strong scaling needs a GPU count that divides %d" % total)
    per = total // world
    return [(u // C_FEAT, u % C_FEAT) for u in range(rank * per, (rank + 1) * per)]


def run_gpu(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the CKKS engine has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    pkg = importlib.import_module(PKG)
    pkg.build()
    eng = pkg.load_engine()
    client = importlib.import_module(PKG + ".client")
    lr = importlib.import_module(PKG + ".lr")
    par = importlib.import_module(PKG + ".parallel")

    primes = _primes()
    ctx = eng.Context(LOG_N, primes, device=local)
    ev = eng.Evaluator(ctx)
    enc = client.CKKSEncoder(ctx)
    kg = client.KeyGenerator(ctx, seed=1234)          # same keys on every rank (one client)
    keys = kg.keyset(steps=[1, -B_MINI])
    fast_steps = []
    while not (args.no_fast or args.ncu) and (1 << len(fast_steps)) < B_MINI:
        fast_steps.append(1 << len(fast_steps))
    keys_fast = kg.keyset(steps=[-B_MINI] + fast_steps) if fast_steps else None
    encr = client.Encryptor(ctx, kg.public_key(), seed=100 + rank)
    decr = client.Decryptor(ctx, kg.secret_key())
    slots = ctx.n // 2
    M = R_PER_GPU // B_MINI
    lay = lr.ColumnLayout(R_PER_GPU, C_FEAT, B_MINI, slots)
    w0 = np.random.default_rng(5).uniform(-1, 1, C_FEAT)
    wvec = np.zeros(slots)
    wvec[:C_FEAT] = w0
    strong = args.scaling == "strong"

    class Problem:
        """client side (untimed): encode + encrypt this rank's part of a problem, resident on the device and as
        PINNED host copies for the e2e leg"""

        def __init__(self, X, y, units, R_total):
            self.X, self.y, self.R_total = X, y, R_total
            ms = sorted({m for m, _ in units})                     # mini-batches this rank touches
            pos = {m: k for k, m in enumerate(ms)}
            self.units = None if len(units) == len(ms) * C_FEAT else [(pos[m], j) for m, j in units]
            self.n_units = len(units)
            colv, labv = lay.columns(X), lay.labels(y)
            rows = [m * C_FEAT + j for m in ms for j in range(C_FEAT)]
            self.cols = encr.encrypt(enc.encode(colv[rows], SCALE))
            self.labs = encr.encrypt(enc.encode(labv[ms], SCALE))
            self.wb = encr.encrypt(enc.encode(np.repeat(w0[:, None], slots, axis=1), SCALE))
            self.w = encr.encrypt(enc.encode(wvec, SCALE))
            self.host = {k: getattr(self, k).data.cpu().pin_memory() for k in ("cols", "labs", "wb", "w")}
            self.h2d_bytes = sum(t.numel() * 8 for t in self.host.values())

        def epoch(self, cols, labs, wb, wct, k=None, dot_method="reference"):
            # all-gather of the partial gradient ciphertexts + mod-q add kernel, before the final rescale (bit-identical
            # to the unsharded epoch)
            grad = lr.column_epoch_gradient(ev, cols, labs, wb, C_FEAT, B_MINI, SCALE, k or keys, enc, encr,
                                            degree=DEGREE, method="tree", dot_method=dot_method, units=self.units,
                                            combine=lambda g: par.combine_partials(ev, g))
            return grad, lr.apply_gradient(ev, grad, wct, LR, self.R_total, SCALE, enc)

        def resident(self):
            return self.epoch(self.cols, self.labs, self.wb, self.w)

        def fast(self):
            # SURVEY 8(f4): the same epoch with the rotate-and-sum of cipher_dot_product done by log2(B)
            # doubling rotations.  Not the reference's op sequence (ciphertexts differ, decrypted results
            # agree within noise): reported beside the headline, never as it.
            return self.epoch(self.cols, self.labs, self.wb, self.w, keys_fast, "doubling")

        def e2e(self, out_host):
            dev = {k: t.to(ctx.device, non_blocking=True) for k, t in self.host.items()}
            top = ctx.top_limbs
            grad, neww = self.epoch(eng.Ciphertext(ctx, dev["cols"], top, SCALE), eng.Ciphertext(ctx, dev["labs"], top, SCALE),
                                    eng.Ciphertext(ctx, dev["wb"], top, SCALE), eng.Ciphertext(ctx, dev["w"], top, SCALE))
            out_host[:, :, : neww.limbs].copy_(neww.data[:, :, : neww.limbs], non_blocking=True)
            return grad, neww

    all_units = [(m, j) for m in range(M) for j in range(C_FEAT)]
    if strong:
        X, y = synthetic_shard(seed=10)                # the same problem on every rank
        prob = Problem(X, y, strong_units(rank, world), R_PER_GPU)
        want = lr.plain_epoch(X, y, w0, LR, DEGREE)
    else:
        X, y = synthetic_shard(seed=10 + rank)
        prob = Problem(X, y, all_units, R_PER_GPU * world)
        shards = [synthetic_shard(seed=10 + r) for r in range(world)] if rank == 0 else [(X, y)]
        want = lr.plain_epoch(np.concatenate([a for a, _ in shards]), np.concatenate([b for _, b in shards]), w0, LR, DEGREE)
    ctx.reserve(prob.n_units, ctx.top_limbs)
    if os.environ.get("CKKS_CHAIN_LANES"):
        ctx.set_chain_lanes(int(os.environ["CKKS_CHAIN_LANES"]))
    out_host = torch.empty((1, 2, ctx.top_limbs, ctx.n), dtype=torch.int64).pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, warmup, steps):
        for _ in range(warmup):
            fn()
        barrier()
        ctx.reset_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.time()
        e0.record()
        for _ in range(steps):
            res = fn()
        e1.record()
        barrier()
        t1 = time.time()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=ctx.device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, res, ctx.launch_count(), t0, t1

    def check(neww, want_w):
        """correctness gate on the timed computation, at every N: decrypted weights vs plaintext LR on the whole data"""
        got = enc.decode(decr.decrypt(neww))[0, :C_FEAT]
        err = float(np.abs(got - want_w).max())
        assert err < 1e-3, "decrypted weights differ from plaintext LR by %g" % err
        return got, err

    sampler = ClockSampler(local) if rank == 0 else None
    if args.ncu:
        for _ in range(args.warmup):
            prob.resident()
        torch.cuda.synchronize()
        torch.cuda.profiler.start()       # ncu --profile-from-start off: capture the timed region only
        prob.resident()
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        return
    ms, (grad, neww), launches, t0, t1 = timed(prob.resident, args.warmup, args.steps)
    clocks = sampler.stop(t0, t1) if sampler else None
    problems_per_step = 1 if strong else world
    value = problems_per_step * args.steps / (ms / 1e3)
    got, err = check(neww, want) if rank == 0 else (None, None)
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, grad, neww, got)

    e2e_steps = args.steps
    ms_e2e, (_, neww_e2e), _, _, _ = timed(lambda: prob.e2e(out_host), 1, e2e_steps)
    value_e2e = problems_per_step * e2e_steps / (ms_e2e / 1e3)
    if rank == 0:
        check(neww_e2e, want)

    fast = None
    if keys_fast is not None:
        ms_fast, (_, neww_fast), launches_fast, _, _ = timed(prob.fast, 2, args.steps)
        fast = {"value": problems_per_step * args.steps / (ms_fast / 1e3), "unit": UNIT, "ms_per_step": ms_fast / args.steps,
                "gpu_launches_per_step_per_gpu": int(launches_fast) // args.steps,
                "note": "rotate-and-sum by log2(%d) doubling rotations instead of the reference's %d unit rotations "
                        "(SURVEY 8 f4): NOT the reference's op sequence, ciphertexts are not bit-identical, decrypted "
                        "weights agree within noise; reported for information, the headline value is the reference "
                        "sequence" % (B_MINI, B_MINI - 1)}
        if rank == 0:
            got_fast = enc.decode(decr.decrypt(neww_fast))[0, :C_FEAT]
            fast["max_abs_diff_vs_reference_sequence"] = float(np.abs(got_fast - got).max())

    # ---- the other scaling mode beside the headline (N > 1): every GPU its own 8 x 32768 shard
    weak = None
    if world > 1 and strong and not args.no_weak:
        Xw, yw = synthetic_shard(seed=10 + rank)
        probw = Problem(Xw, yw, all_units, R_PER_GPU * world)
        ms_w, (_, neww_w), _, _, _ = timed(probw.resident, 1, args.steps)
        weak = {"value": world * args.steps / (ms_w / 1e3), "unit": UNIT, "scaling": "weak", "ms_per_step": ms_w / args.steps, "steps": args.steps,
                "note": "every GPU holds its own 8 x 32768 shard (N independent problems, one combined update)"}
        if rank == 0:
            sh = [synthetic_shard(seed=10 + r) for r in range(world)]
            want_w = lr.plain_epoch(np.concatenate([a for a, _ in sh]), np.concatenate([b for _, b in sh]), w0, LR, DEGREE)
            weak["max_abs_err_vs_plaintext_lr"] = check(neww_w, want_w)[1]
        del probw

    # ---- config 3 beside the headline: Linear_Transform_Plain, N = 16384, d = 128, diagonals sharded
    # over the ranks (interleaved), partial ciphertexts all-gathered and added mod q.  Strong scaling.
    lt = None
    if not args.no_lt:
        lt = linear_transform_sharded(torch, eng, client, par, local, rank, world, timed)

    # ---- roofline of the dominant kernel family: the batched Galois key switch of the dot-product
    # chain (M*C = 32 ciphertexts, L = 3) -- one launch group = 5 fused kernels per lane, timed live with CUDA
    # events on the launching stream (torch's current stream; the engine forks/joins its lane streams on it)
    Lk = ctx.top_limbs - 6
    nb = M * C_FEAT
    a = ctx.empty(nb, 2, Lk, cap=ctx.top_limbs, scale=SCALE)
    a.data.random_(0, 1 << 39)
    b = a.like()
    g1 = ctx.galois_elt(1)
    for _ in range(5):
        ev.apply_galois(a, g1, keys, out=b)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 200
    e0.record()
    for _ in range(reps // 2):
        ev.apply_galois(a, g1, keys, out=b)
        ev.apply_galois(b, g1, keys, out=a)
    e1.record()
    torch.cuda.synchronize()
    ks_ms = e0.elapsed_time(e1) / reps
    alg = nb * ks_bytes(Lk, ctx.n)
    peak, peak_src = peaks()
    achieved = alg / (ks_ms * 1e-3) / 1e9
    prof = {}
    tpath = os.path.join(ROOT, "profiles", "keyswitch_traffic.json")
    if os.path.exists(tpath):
        prof = json.load(open(tpath))
    # the same figure from the timed epochs themselves: every epoch of this GPU is prob.n_units chains of B_MINI Galois
    # key switches at L = 3 (99.9 % of its launches), so algorithmic bytes / step time cross-checks the micro-measurement
    epoch_alg = prob.n_units * B_MINI * ks_bytes(Lk, ctx.n)
    roofline = {
        "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
        "traffic": prof.get("bytes_per_launch_group"), "traffic_source": prof.get("source"),
        "kernel": "Galois key switch launch group (k_ks_intt_row, k_ks_invcol_modup, k_ks_mac + k_ks_mac_fp, "
                  "k_md_invcol_fwdcol, k_md_fwd_row), batch %d, N=32768, L=%d" % (nb, Lk),
        "algorithmic_bytes_per_launch_group": alg, "ms_per_launch_group": ks_ms, "peak_source": peak_src,
        "keyswitch_per_s": nb / (ks_ms * 1e-3),
        "from_timed_epochs": {"achieved": epoch_alg / (ms / args.steps * 1e-3) / 1e9,
                              "frac": epoch_alg / (ms / args.steps * 1e-3) / 1e9 / peak,
                              "keyswitches_per_step_per_gpu": prob.n_units * B_MINI},
        "pipe_utilisation": prof.get("pipe_utilisation"),
        "arithmetic_ceiling": arithmetic_ceiling(Lk, ks_ms * 1e3 / nb),
        "note": "HBM is the roofline north_star names; the key switch does L^2+3L+2 = 20 size-N NTTs per 9.4 MB, so issue "
                "slots and the integer-multiplier / FP64 pipes bind before HBM (DESIGN.md section 4; pipe_utilisation = ncu "
                "sm__inst_executed_pipe_* of the same launch group, profiles/)",
    }
    ks_extra = keyswitch_sweep(torch, eng, ctx, ev, keys) if rank == 0 and not args.no_sweep else None
    ops = op_rooflines(torch, eng, ctx, ev) if rank == 0 and not args.no_sweep else None

    cfg1 = None
    if rank == 0 and world == 1 and not args.no_config1:
        del a, b
        cfg1 = config1_pulsar(torch, eng, client, lr, ctx, ev, enc, kg, encr, decr, timed)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = cpu_reference(budget_s=args.cpu_budget)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "u64", "data": "synthetic", "config": workload_config(world, args.scaling),
            "e2e": {"value": value_e2e, "unit": UNIT, "h2d_bytes_per_step": prob.h2d_bytes,
                    "d2h_bytes_per_step": int(out_host[:, :, : neww.limbs].numel() * 8), "steps": e2e_steps,
                    "ms_per_step": ms_e2e / e2e_steps},
            "gpu_launches": int(launches) * world,
            "gpu_launches_per_step_per_gpu": int(launches) // args.steps,
            "gradient_units_per_gpu": prob.n_units,
            "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
            "keyswitch_ops_per_s": ks_extra, "op_rooflines": ops, "weak_scaling": weak, "doubling_mode": fast,
            "linear_transform": lt, "config1_pulsar": cfg1,
            "check": {"max_abs_err_vs_plaintext_lr": err, "tolerance": 1e-3,
                      "what": "decrypted updated weights of the timed epoch (resident and e2e legs) vs plaintext LR on the whole data, at every N"},
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def op_rooflines(torch, eng, ctx15, ev15):
    """element-wise ops and rescale against the HBM roofline (algorithmic bytes of SURVEY.md 8(d): add 48 L N,
    multiply_plain 40 L N, multiply 56 L N, rescale 8 S (2L-1) N), batches larger than L2, CUDA events"""
    params = importlib.import_module(PKG + ".params")
    peak, _ = peaks()
    out = {}
    for log_n, bits, batch in ((14, [60] + [40] * 7 + [60], 512), (15, BITS, 256)):
        ctx = ctx15 if log_n == 15 else eng.Context(log_n, params.coeff_modulus_create(log_n, bits))
        ev = ev15 if log_n == 15 else eng.Evaluator(ctx)
        L, n = ctx.top_limbs, ctx.n
        a = ctx.empty(batch, 2, L, scale=SCALE)
        a.data.random_(0, 1 << 39)
        b = a.clone()
        pt = ctx.empty(batch, 1, L, scale=SCALE)
        pt.data.random_(0, 1 << 39)
        o2, o3 = a.like(), a.like(size=3)
        cases = (("add", lambda: ev.add(a, b, out=o2), 48 * L * n),
                 ("multiply_plain", lambda: ev.multiply_plain(a, pt, out=o2), 40 * L * n),
                 ("multiply", lambda: ev.multiply(a, b, out=o3), 56 * L * n),
                 ("rescale_to_next", lambda: ev.rescale_to_next(a, out=o2), 8 * 2 * (2 * L - 1) * n))
        res = {}
        for name, fn, nbytes in cases:
            a.scale = b.scale = pt.scale = 1.0
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 10
            e0.record()
            for _ in range(reps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            msr = e0.elapsed_time(e1) / reps
            gbs = batch * nbytes / (msr * 1e-3) / 1e9
            res[name] = {"ops_per_s": batch / (msr * 1e-3), "batch": batch, "achieved_gbs": gbs, "frac_of_hbm_peak": gbs / peak}
        out["N=%d,L=%d" % (n, L)] = res
        del a, b, pt, o2, o3
    return out


def config1_pulsar(torch, eng, client, lr, ctx, ev, enc, kg, encr, decr, timed):
    """BASELINE configs[0]: the reference's own LR program (row layout, Horner degree-3 sigmoid, lr 0.1,
    logistic_regression_ckks.cpp:208-345 with the repairs of lr.py) on the first 2000 rows of pulsar_stars.csv
    (tests/golden copy of the reference's file), standardised with the reference's scaler, starting from the reference
    program's own initial weights.  N = 32768, {60, 40 x 8, 60}: the chain the file names (N = 16384, {60,40x7,60};
    BASELINE.json says 8192) cannot hold one iteration (SURVEY 3.4-2).  One step = one update_weights (training
    iteration) over all 2000 rows; checked against plaintext LR with the same polynomial."""
    pulsar = importlib.import_module(PKG + ".pulsar")
    gold_path = os.path.join(ROOT, "tests", "golden", "pulsar_plain_lr.json")
    if not (os.path.exists(pulsar.DEFAULT_CSV) and os.path.exists(gold_path)):
        return {"unavailable": "tests/golden/pulsar_stars.csv missing"}
    gold = json.load(open(gold_path))
    X, y = pulsar.load_csv()
    Xs, y = pulsar.standard_scaler(X).astype(np.float64), y.astype(np.float64)
    w0 = np.array(gold["initial_weights"])
    R, C = Xs.shape
    keys = kg.keyset(steps=[s for i in range(13) for s in (1 << i, -(1 << i))])
    lay = lr.RowLayout(R, C, ctx.n // 2)
    rows = encr.encrypt(enc.encode(lay.rows(Xs), SCALE))
    cols = encr.encrypt(enc.encode(lay.columns(Xs), SCALE))
    labs = encr.encrypt(enc.encode(lay.labels(y), SCALE))
    wct = encr.encrypt(enc.encode(lay.weights(w0), SCALE))
    ms, neww, launches, _, _ = timed(lambda: lr.update_weights(ev, rows, cols, labs, wct, LR, SCALE, keys, enc, encr, degree=3,
                                                               method="horner"), 1, 2)
    got = enc.decode(decr.decrypt(neww))[0, :C]
    want = lr.plain_epoch(Xs, y, w0, LR, 3)
    return {"workload": "update_weights on pulsar_stars.csv (2000 x 8, standardised), row layout, Horner degree 3, N=32768 {60,40x8,60}",
            "ms_per_iteration": ms / 2, "iterations_per_s": 2e3 / ms, "gpu_launches_per_iteration": int(launches) // 2,
            "key_switches_per_iteration": R * (1 + 1 + C - 1) + C * (1 + 13 + R - 1) + 3,
            "max_abs_err_vs_plaintext_polynomial_lr": float(np.abs(got - want).max()),
            "max_abs_diff_vs_reference_program_true_sigmoid_step": float(np.abs(got - np.array(gold["weights_after_iteration_0"])).max()),
            "cost_after_step": pulsar.cost_function(Xs.astype(np.float32), y, got),
            "reference_program_cost_after_iteration_0": gold["cost_after_iteration_0"]}


def linear_transform_sharded(torch, eng, client, par, local, rank, world, timed, d=128, log_n=14):
    """BASELINE config 3 (linear_transformation2.cpp, helper.h:237-262) with the diagonals sharded
    across the ranks (SURVEY 8(e)): every rank rotates ct + rot(ct,-d) by ITS diagonals' steps,
    multiplies by its plaintext diagonals and sums; one all-gather + mod-q add combines the partial
    ciphertexts.  The combined ciphertext is checked bit-for-bit against the unsharded transform."""
    wl = importlib.import_module(PKG + ".workloads")
    params = importlib.import_module(PKG + ".params")
    ctx = eng.Context(log_n, params.coeff_modulus_create(log_n, [60, 40, 40, 60]), device=local)
    ev = eng.Evaluator(ctx)
    enc = client.CKKSEncoder(ctx)
    kg = client.KeyGenerator(ctx, seed=77)               # same keys and inputs on every rank
    keys = kg.keyset(steps=[s for i in range(8) for s in (1 << i, -(1 << i))])
    encr = client.Encryptor(ctx, kg.public_key(), seed=78)
    decr = client.Decryptor(ctx, kg.secret_key())
    rng = np.random.default_rng(79)
    U, v = rng.uniform(0, 1, (d, d)), rng.uniform(0, 1, d)
    ct = encr.encrypt(enc.encode(v, SCALE))
    diags = enc.encode(wl.all_diagonals(U), SCALE)
    plans = wl.PlanCache(ctx, keys)
    mine = par.shard_rotations_shared(list(range(d)), rank, world)   # neighbours in NAF-prefix order, balanced by key switches
    idx = torch.tensor(mine, device=ctx.device)
    diags_local = eng.Ciphertext(ctx, diags.data[idx].contiguous(), diags.limbs, diags.scale)

    def sharded():
        dup = wl.duplicate_fill(ev, ct, d, keys)
        return par.sharded_linear_transform_plain(ev, lambda steps: ev.rotate_plan(dup, plans.get(steps)), diags_local, d, mine)

    full = wl.linear_transform_plain(ev, ct, diags, keys, plans)
    bsgs = None
    if world == 1:   # SURVEY 8(f4) mode beside it: baby-step / giant-step, tolerance-checked, not the reference sequence
        bd = wl.BsgsDiagonals(U, SCALE, enc, baby=16)
        ms_b, out_b, _, _, _ = timed(lambda: wl.linear_transform_plain_bsgs(ev, ct, bd, keys, plans), 3, 20)
        bsgs = {"ms": ms_b / 20, "baby": bd.b, "giant": bd.G,
                "key_switches": int(plans.get(range(bd.b)).keyswitches + plans.get([g * bd.b for g in range(bd.G)]).keyswitches + 1),
                "max_abs_err_vs_plain": float(np.abs(enc.decode(decr.decrypt(out_b))[0, :d] - U @ v).max()),
                "note": "not the reference's op sequence; ciphertexts differ, decrypted result agrees"}
    hoisted = None
    if world == 1:   # SURVEY 8(f4) mode beside it: hoisted rotations (one digit decomposition shared by all d-1 rotations)
        keys_h = kg.keyset(steps=[-d] + list(range(1, d)), relin=False)        # a Galois key for every step itself
        plans_h = wl.PlanCache(ctx, keys_h)
        ms_h, out_h, _, _, _ = timed(lambda: wl.linear_transform_plain_hoisted(ev, ct, diags, keys_h, plans_h), 3, 20)
        # with those keys SEAL's own rotate_vector needs ONE key switch per rotation (no NAF chain): the reference sequence
        # itself, bit-exact for this key set, 128 instead of 356 key switches in one round
        ms_d, out_d, _, _, _ = timed(lambda: wl.linear_transform_plain(ev, ct, diags, keys_h, plans_h), 3, 20)
        bdh = wl.BsgsDiagonals(U, SCALE, enc, baby=16)
        ms_bh, out_bh, _, _, _ = timed(lambda: wl.linear_transform_plain_bsgs_hoisted(ev, ct, bdh, keys_h, plans_h), 3, 20)
        hoisted = {"ms": ms_h / 20, "key_switch_inner_products": d, "full_key_switches": 1, "galois_keys": d,
                   "max_abs_err_vs_plain": float(np.abs(enc.decode(decr.decrypt(out_h))[0, :d] - U @ v).max()),
                   "bsgs_hoisted_ms": ms_bh / 20,
                   "reference_sequence_with_direct_keys_ms": ms_d / 20,
                   "reference_sequence_with_direct_keys_max_abs_err": float(np.abs(enc.decode(decr.decrypt(out_d))[0, :d] - U @ v).max()),
                   "bsgs_hoisted_max_abs_err_vs_plain": float(np.abs(enc.decode(decr.decrypt(out_bh))[0, :d] - U @ v).max()),
                   "note": "not the reference's op sequence (SEAL permutes before lifting digits): ciphertexts differ, decrypted "
                           "result agrees within key-switch noise; needs one Galois key per step instead of SEAL's default 2 log2 N"}
        del keys_h, plans_h
    ms_eager, out, _, _, _ = timed(sharded, 3, 20)
    # the transform is ~40 short launches per GPU (<= 4 dependent NAF rounds) + one all-gather: at 8 GPUs the host launch
    # path, not the GPU, sets the pace.  Capture the whole sharded transform (rotation rounds, fused products, NCCL
    # all-gather, mod-q add) into ONE CUDA graph and replay it.
    ctx.reserve(len(mine), ctx.top_limbs)   # a captured key switch runs as one lane: size the workspace before capturing
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    try:
        with torch.cuda.graph(graph):
            out = sharded()
        ms_graph, _, _, _, _ = timed(graph.replay, 3, 20)
        graphed = {"ms": ms_graph / 20}
        ms = min(ms_graph, ms_eager)      # the replayed graph runs every key switch as one lane: it wins when launches bind (many GPUs)
    except Exception as exc:          # capture unsupported in this environment: keep the eager timing, say so
        ms, graphed = ms_eager, "capture failed: %s" % str(exc)[:120]
        torch.cuda.synchronize()
        out = sharded()
    same = bool(torch.equal(out.data[:, :, : out.limbs], full.data[:, :, : full.limbs]))
    err = float(np.abs(enc.decode(decr.decrypt(out))[0, :d] - U @ v).max())
    ks_local = plans.get(mine).keyswitches_shared + 1
    return {"workload": "Linear_Transform_Plain d=%d, N=%d, {60,40,40,60}, diagonals sharded over %d GPU(s)" % (d, 1 << log_n, world),
            "ms": ms / 20, "transforms_per_s": 20e3 / ms, "scaling": "strong", "key_switches_per_gpu": int(ks_local),
            "key_switches_per_gpu_reference_sequence": int(plans.get(mine).keyswitches + 1),
            "note": "rotations of the one input ciphertext share their common NAF prefixes: fewer key switches, every output "
                    "bit-identical to its own rotate_vector call",
            "cuda_graph": graphed, "ms_eager_launches": ms_eager / 20, "rounds": int(plans.get(mine).rounds),
            "bit_identical_to_unsharded": same, "max_abs_err_vs_plain": err, "bsgs_mode": bsgs, "hoisted_mode": hoisted}


def arithmetic_ceiling(L, us_per_key_switch):
    """the key switch against the measured throughput of its own butterflies (profiles/micro/butterfly_rates.cu: the
    engine's radix-8 register steps on register-resident data, no memory traffic): time the 20 (L = 3) transforms'
    butterflies alone would take on this GPU, and the share of the live-timed key switch that is"""
    path = os.path.join(ROOT, "profiles", "butterfly_rates.json")
    if not os.path.exists(path):
        return None
    doc = json.load(open(path))
    key = "key_switch_N32768_L%d" % L
    if key not in doc:
        return None
    serial = doc[key]["us_butterflies_only_pipes_serial"]
    mixed = doc[key].get("us_butterflies_only_measured_concurrent_mix", serial)
    return {"us_per_key_switch_butterflies_only": mixed, "us_per_key_switch_measured": us_per_key_switch,
            "frac": mixed / us_per_key_switch, "transforms": doc[key]["transforms"], "source": doc["source"],
            "note": "compute ceiling of the butterflies alone (integer and FP64 kernels running concurrently); the inner "
                    "product, reductions, exchanges and memory instructions come on top"}


def _primes():
    """CoeffModulus::Create(32768, {60, 40 x 8, 60}) -- product-side restatement of SEAL's prime
    search (first occurrence of a size gets the smallest of that size's primes)."""
    pkg = importlib.import_module(PKG + ".params")
    return pkg.coeff_modulus_create(LOG_N, BITS)


def keyswitch_sweep(torch, eng, ctx15, ev15, keys15):
    """second half of the metric: rotate / relinearize key-switch ops/s at N = 2^14 and 2^15"""
    client = importlib.import_module(PKG + ".client")
    params = importlib.import_module(PKG + ".params")
    out = {}
    peak, _ = peaks()
    for log_n, bits, batch in ((14, [60, 40, 40, 60], 256), (14, [60] + [40] * 7 + [60], 64), (15, BITS, 32)):
        if log_n == 15:
            ctx, ev, keys = ctx15, ev15, keys15
        else:
            ctx = eng.Context(log_n, params.coeff_modulus_create(log_n, bits))
            ev = eng.Evaluator(ctx)
            keys = client.KeyGenerator(ctx, seed=3).keyset(steps=[1])
        L = ctx.top_limbs
        a = ctx.empty(batch, 2, L, scale=SCALE)
        a.data.random_(0, 1 << 39)
        a3 = ctx.empty(batch, 3, L, scale=SCALE)
        a3.data.random_(0, 1 << 39)
        b, b2 = a.like(), a.like()
        g1 = ctx.galois_elt(1)
        res = {}
        for name, fn, relin in (("rotate", lambda: ev.apply_galois(a, g1, keys, out=b), False),
                                ("relinearize", lambda: ev.relinearize(a3, keys, out=b2), True)):
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 20
            e0.record()
            for _ in range(reps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / reps
            gbs = batch * ks_bytes(L, ctx.n, relin) / (ms * 1e-3) / 1e9
            res[name] = {"ops_per_s": batch / (ms * 1e-3), "batch": batch, "achieved_gbs": gbs, "frac_of_hbm_peak": gbs / peak}
        out["N=%d,L=%d" % (ctx.n, L)] = res
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3,
                    help="timed epochs of every config-5 epoch leg (headline, e2e, doubling mode, weak scaling); the "
                         "config-1, linear-transform and key-switch sweep legs time fixed repetition counts")
    ap.add_argument("--warmup", type=int, default=3,
                    help="untimed epochs before the headline leg; the later legs warm up with their own fixed counts "
                         "(1 to 3 calls)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-sweep", action="store_true", help="skip the key-switch ops/s sweep")
    ap.add_argument("--cpu-budget", type=float, default=20.0)
    ap.add_argument("--no-lt", action="store_true", help="skip the sharded linear-transform (config 3) leg")
    ap.add_argument("--no-fast", action="store_true", help="skip the informational doubling-mode epoch")
    ap.add_argument("--ncu", action="store_true", help="profiling run: one epoch between cudaProfilerStart/Stop, no JSON")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong: one 8 x 32768 problem split over the GPUs (default, BASELINE config 5); weak: one shard per GPU")
    ap.add_argument("--no-weak", action="store_true", help="skip the weak-scaling leg reported beside the strong one at N > 1")
    ap.add_argument("--no-config1", action="store_true", help="skip the config-1 (pulsar CSV) leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed epoch computed to DIR/<name>.npy (float64); inputs, keys and encryption "
                         "randomness are seeded, so runs with the same arguments write the same arrays and two builds can "
                         "be compared output for output")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.ncu and args.dump_outputs:
        ap.error("--dump-outputs needs the timed epochs, which --ncu does not run")
    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        # started as plain `python bench.py --gpus N`: relaunch as one process per GPU
        import socket
        with socket.socket() as sock:
            sock.bind(("127.0.0.1", 0))
            port = sock.getsockname()[1]
        os.execvp(sys.executable, [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
                                   "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.abspath(__file__)] + sys.argv[1:])
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
