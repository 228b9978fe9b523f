"""Strong scaling of the double-hoisted workloads sharded with parallel.sharded_* over the GPUs of one node:
config 3 (N = 16384, {60, 40, 40, 60}) linear transform at d = 64 and d = 128, one-output and BSGS, and config 4
(N = 16384, {60, 40 x 4, 60}) 64 x 64 product, against the one-GPU double-hoisted functions in the same run.

    python -m torch.distributed.run --nproc_per_node G profiles/double_hoisting_scaling.py [--reps 20] [--out-dir DIR]

Rank 0 writes DIR/r09_double_hoisting_scaling_<G>gpu.json.  Per workload: the median of alternated sharded and one-GPU
calls (host clock around a call ended by a device synchronise; the sharded time is the slowest rank's), the phases of
the sharded call from CUDA events on rank 0 (partial, exchange, mod_down, and for the product step2 and tail), counted
key inner products per rank, bytes each rank sends, Galois keys each rank needs (and their bytes), bit-identity with
the one-GPU ciphertext, and the GPU's name and power limit read in the same run.  Every rank loads the one-GPU key set
(same seed on every rank, so that the one-GPU reference is the same ciphertext); the keys a rank needs are counted."""
import argparse
import importlib
import json
import os
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))
from matmul_scaling import CountingExchange, gpu_info  # noqa: E402

PKG = "seal-fyp-logistic-regression_b200"
SCALE, EPS = 2.0 ** 40, 1e-8


class Phases:
    """CUDA events at the sharded call's phase marks; elapsed milliseconds per phase"""

    def __init__(self):
        self.events = []

    def start(self):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        self.events = [("start", e)]

    def __call__(self, name):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        self.events.append((name, e))

    def ms(self):
        return {n: a[1].elapsed_time(b) for a, (n, b) in zip(self.events, self.events[1:])}


def timed(fn, sync_all):
    torch.cuda.synchronize()
    if sync_all:
        dist.barrier()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, (time.perf_counter() - t0) * 1e3


def measure(name, sharded, one_gpu, reps, warmup, ctx, extra):
    """alternated sharded / one-GPU calls; sharded time = slowest rank"""
    rank, world = dist.get_rank(), dist.get_world_size()
    ph = Phases()
    ts, tu, phases = [], [], []
    for i in range(warmup + reps):
        ph.start()
        out, t = timed(lambda: sharded(ph), True)
        torch.cuda.synchronize()
        tt = torch.tensor([t], device=ctx.device)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        want, u = timed(one_gpu, False)
        if i >= warmup:
            ts.append(float(tt.item()))
            tu.append(u)
            phases.append(ph.ms())
    same = bool(out.limbs == want.limbs and out.scale == want.scale and out.size == want.size
                and torch.equal(out.data[:, :, :out.limbs], want.data[:, :, :want.limbs]))
    flags = torch.tensor([int(same)], device=ctx.device)
    dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    med = {k: float(np.median([p[k] for p in phases])) for k in phases[0]}
    res = {"workload": name, "ms_sharded": float(np.median(ts)), "ms_sharded_all": ts,
           "ms_one_gpu": float(np.median(tu)), "ms_one_gpu_all": tu,
           "phases_ms_rank0_median": med, "bit_identical_on_every_rank": bool(flags.item())}
    res.update(extra)
    return res, out


def per_rank(values, ctx):
    t = torch.tensor(values, device=ctx.device, dtype=torch.int64)
    allv = [torch.zeros_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(allv, t)
    return [[int(x) for x in v.tolist()] for v in allv]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out-dir", default=".")
    args = ap.parse_args()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()
    eng = importlib.import_module(PKG).load_engine()
    wl, par = importlib.import_module(PKG + ".workloads"), importlib.import_module(PKG + ".parallel")
    client, params = importlib.import_module(PKG + ".client"), importlib.import_module(PKG + ".params")
    results = []

    # ---- config 3: linear transforms
    ctx = eng.Context(14, params.coeff_modulus_create(14, [60, 40, 40, 60]), device=local)
    ev, enc = eng.Evaluator(ctx), client.CKKSEncoder(ctx)
    kg = client.KeyGenerator(ctx, seed=11)
    steps = set()
    for d in (64, 128):
        steps |= set(wl.linear_transform_double_hoisted_steps(d)) | set(wl.bsgs_double_hoisted_steps(d, int(round(d ** 0.5))))
    keys = kg.keyset(steps=sorted(steps), relin=False)
    key_bytes = (ctx.K - 1) * 2 * ctx.K * ctx.n * 8
    encr, decr = client.Encryptor(ctx, kg.public_key(), seed=12), client.Decryptor(ctx, kg.secret_key())
    plans = wl.PlanCache(ctx, keys)
    for d in (64, 128):
        rng = np.random.default_rng(d)
        U, v = rng.uniform(0, 1, (d, d)), rng.uniform(0, 1, d)
        ct = encr.encrypt(enc.encode(v, SCALE))
        diags = enc.encode(wl.all_diagonals(U), SCALE, limbs=ctx.K)
        bd = wl.BsgsDiagonals(U, SCALE, enc, limbs=ctx.K)
        for kind in ("one-output", "bsgs"):
            ex = CountingExchange(par)
            if kind == "one-output":
                mine = par.shard_terms(wl.diagonal_terms([range(d)], [0]), rank, world)
                ips = sum(1 for t in mine[0] if t[1] != 0)
                nkeys = len(par.linear_transform_double_hoisted_rank_steps(d, rank, world))
                sharded = lambda ph: par.sharded_linear_transform_plain_double_hoisted(ev, ct, diags, keys, plans, rank,
                                                                                       world, ex, mark=ph)
                one = lambda: wl.linear_transform_plain_double_hoisted(ev, ct, diags, keys, plans)
            else:
                own, baby, giant = par._bsgs_rank_tables(d, bd.b, rank, world)
                ips = sum(1 for terms in baby + (giant[0:1] if giant else []) for t in terms if t[1] != 0)
                nkeys = len(par.bsgs_double_hoisted_rank_steps(d, bd.b, rank, world))
                sharded = lambda ph: par.sharded_linear_transform_plain_bsgs_double_hoisted(ev, ct, bd, keys, plans, rank,
                                                                                            world, ex, mark=ph)
                one = lambda: wl.linear_transform_plain_bsgs_double_hoisted(ev, ct, bd, keys, plans)
            res, out = measure("config 3 linear transform d=%d, %s, double hoisted" % (d, kind), sharded, one,
                               args.reps, args.warmup, ctx, {})
            sent = ex.sent // (args.reps + args.warmup)
            counts = per_rank([ips, sent, nkeys], ctx)
            res.update(inner_products_per_rank=[c[0] for c in counts], bytes_sent_per_rank=[c[1] for c in counts],
                       galois_keys_per_rank=[c[2] for c in counts], galois_key_bytes_per_rank=[c[2] * key_bytes for c in counts],
                       max_abs_err_vs_Uv=float(np.abs(enc.decode(decr.decrypt(out))[0, :d] - U @ v).max()))
            results.append(res)
    del keys, plans

    # ---- config 4: 64 x 64 product
    D = 64
    ctx4 = eng.Context(14, params.coeff_modulus_create(14, [60, 40, 40, 40, 40, 60]), device=local)
    ev4, enc4 = eng.Evaluator(ctx4), client.CKKSEncoder(ctx4)
    kg4 = client.KeyGenerator(ctx4, seed=21)
    keys4 = kg4.keyset(steps=wl.matmul_nonzero_hoisted_steps(D))
    key_bytes4 = (ctx4.K - 1) * 2 * ctx4.K * ctx4.n * 8
    encr4, decr4 = client.Encryptor(ctx4, kg4.public_key(), seed=22), client.Decryptor(ctx4, kg4.secret_key())
    plans4 = wl.PlanCache(ctx4, keys4)
    rng = np.random.default_rng(4)
    A, B = rng.uniform(0, 1, (D, D)), rng.uniform(0, 1, (D, D))
    mk = lambda U: wl.DiagonalSet.from_matrix(U, EPS, SCALE, enc4, limbs=ctx4.K)
    sig, tau = mk(wl.u_sigma(D)), mk(wl.u_tau(D))
    V = [mk(wl.v_k(D, k)) for k in range(1, D)]
    W = [mk(wl.w_k(D, k)) for k in range(1, D)]
    ctA, ctB = encr4.encrypt(enc4.encode(A.reshape(-1), SCALE)), encr4.encrypt(enc4.encode(B.reshape(-1), SCALE))
    first, own, second = par._matmul_rank_tables(sig.index, tau.index, [s.index for s in V], [s.index for s in W], rank, world)
    ips = sum(1 for tbl in (first, second) for terms in tbl for t in terms if t[1] != 0)
    ex = CountingExchange(par)
    res, out = measure("config 4 64x64 product, nonzero diagonals, double hoisted",
                       lambda ph: par.sharded_cc_matrix_multiplication_nonzero_hoisted(ev4, ctA, ctB, D, sig, tau, V, W,
                                                                                      keys4, plans4, rank, world, ex,
                                                                                      mark=ph),
                       lambda: wl.cc_matrix_multiplication_nonzero_hoisted(ev4, ctA, ctB, D, sig, tau, V, W, keys4, plans4),
                       args.reps, args.warmup, ctx4, {})
    counts = per_rank([ips, ex.sent // (args.reps + args.warmup), len(par.matmul_nonzero_hoisted_rank_steps(D, rank, world))],
                      ctx4)
    dec = enc4.decode(decr4.decrypt(out))[0, :D * D].reshape(D, D)
    res.update(inner_products_per_rank=[c[0] for c in counts], bytes_sent_per_rank=[c[1] for c in counts],
               galois_keys_per_rank=[c[2] for c in counts], galois_key_bytes_per_rank=[c[2] * key_bytes4 for c in counts],
               max_abs_err_vs_AB=float(np.abs(dec - A @ B).max()))
    results.append(res)

    if rank == 0:
        rec = {"gpus": world, "gpu": gpu_info(local),
               "timing": "medians of %d alternated sharded / one-GPU calls after %d warm-up pairs; host clock ended by a "
                         "device synchronise, sharded = slowest rank; phases from CUDA events on rank 0" % (args.reps, args.warmup),
               "results": results}
        os.makedirs(args.out_dir, exist_ok=True)
        path = os.path.join(args.out_dir, "r09_double_hoisting_scaling_%dgpu.json" % world)
        json.dump(rec, open(path, "w"), indent=1)
        for r in results:
            print(json.dumps({k: r[k] for k in ("workload", "ms_sharded", "ms_one_gpu", "bit_identical_on_every_rank",
                                                "phases_ms_rank0_median", "inner_products_per_rank")}), flush=True)
        print("wrote", path, flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
