"""Strong scaling of the encrypted 64 x 64 matrix product (BASELINE config 4, CC_Matrix_Multiplication, d = 64,
N = 16384, {60,40,40,40,40,60}, power-of-two Galois keys; the set-up of profiles/run_configs.py: config4) sharded with
parallel.sharded_cc_matrix_multiplication over the GPUs of one node.

    python -m torch.distributed.run --nproc_per_node G profiles/matmul_scaling.py [--reps 5] [--warmup 1] [--out-dir DIR]

Rank 0 writes DIR/r03_matmul_scaling_<G>gpu.json (DIR defaults to the current directory): milliseconds per product
(host clock around the product, ended by a device synchronise on every rank; the slowest rank per repetition), key
switches per GPU, bytes exchanged per rank, the achieved bandwidth of ckks_add_many_grouped at this G's reduce-scatter
shape, bit-identity with the one-GPU cc_matrix_multiplication_sparse (rank 0 also times it), max |decrypt - A @ B|,
and the GPU's name and power limit read in the same run."""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
PKG = "seal-fyp-logistic-regression_b200"
SCALE, EPS, D = 2.0 ** 40, 1e-8, 64
HBM_PEAK_GBS = 7700.0          # NVIDIA HGX B200 data sheet, one GPU


def gpu_info(index):
    info = {"name": torch.cuda.get_device_name(index)}
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit,clocks.max.sm",
                              "--format=csv,noheader,nounits"], stdout=subprocess.PIPE, text=True, timeout=30).stdout
        pl, mx = [x.strip() for x in out.strip().split(",")]
        info.update(power_limit_w=float(pl), sm_max_mhz=float(mx))
    except Exception as exc:      # reported, not guessed
        info.update(power_limit_w=None, power_limit_error=str(exc)[:200])
    return info


class CountingExchange:
    """parallel.TorchExchange that counts the bytes this rank sends to and receives from other ranks"""

    def __init__(self, par):
        self.inner = par.TorchExchange()
        self.rank, self.world = self.inner.rank, self.inner.world
        self.sent = self.received = 0

    def all_gather(self, t):
        nb = t.numel() * t.element_size()
        self.sent += nb * (self.world - 1)
        self.received += nb * (self.world - 1)
        return self.inner.all_gather(t)

    def all_to_all(self, t, send_counts, recv_counts):
        per = t[0].numel() * t.element_size()
        self.sent += per * (sum(send_counts) - send_counts[self.rank])
        self.received += per * (sum(recv_counts) - recv_counts[self.rank])
        return self.inner.all_to_all(t, send_counts, recv_counts)


def grouped_bandwidth(eng, ctx, ev, groups, M, limbs, reps=50):
    """ckks_add_many_grouped at the reduce-scatter shape (groups x M size-2 ciphertexts in, M out); the inputs rotate
    over buffers of 4x the 126 MB L2 so every pass reads HBM"""
    per_in = groups * M * 2 * limbs * ctx.n * 8
    nbuf = max(2, -(-4 * 126 * 2 ** 20 // per_in))
    bufs = [ctx.empty(groups * M, 2, limbs) for _ in range(nbuf)]
    for b in bufs:
        b.data.random_(0, ctx.primes[limbs - 1])
    out = ctx.empty(M, 2, limbs)
    for b in bufs:
        ev.add_many_grouped(b, groups, out=out)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(reps):
        ev.add_many_grouped(bufs[i % nbuf], groups, out=out)
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / reps
    nbytes = (groups + 1) * M * 2 * limbs * ctx.n * 8
    return {"groups": groups, "M": M, "size": 2, "limbs": limbs, "N": ctx.n, "us_per_call": us,
            "algorithmic_bytes": nbytes, "achieved_gbs": nbytes / us * 1e-3,
            "fraction_of_hbm_peak": nbytes / us * 1e-3 / HBM_PEAK_GBS,
            "note": "inputs rotate over %d buffers (%.0f MB, > L2): HBM reads; peak = %.0f GB/s (HGX B200 data sheet)" % (
                nbuf, nbuf * per_in / 2 ** 20, HBM_PEAK_GBS)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out-dir", default=".", help="directory for the JSON (created if missing)")
    args = ap.parse_args()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()

    eng = importlib.import_module(PKG).load_engine()
    wl, par = importlib.import_module(PKG + ".workloads"), importlib.import_module(PKG + ".parallel")
    client, params = importlib.import_module(PKG + ".client"), importlib.import_module(PKG + ".params")
    pow2 = [s for i in range(13) for s in (1 << i, -(1 << i))]
    ctx = eng.Context(14, params.coeff_modulus_create(14, [60, 40, 40, 40, 40, 60]), device=local)
    ev = eng.Evaluator(ctx)
    enc = client.CKKSEncoder(ctx)
    kg = client.KeyGenerator(ctx, seed=5)                  # same keys and inputs on every rank
    keys = kg.keyset(steps=pow2)
    encr = client.Encryptor(ctx, kg.public_key(), seed=6)
    plans = wl.PlanCache(ctx, keys)
    rng = np.random.default_rng(4)
    A, B = rng.uniform(0, 1, (D, D)), rng.uniform(0, 1, (D, D))
    mk = lambda U: wl.DiagonalSet.from_matrix(U, EPS, SCALE, enc)
    sigma, tau = mk(wl.u_sigma(D)), mk(wl.u_tau(D))
    V = [mk(wl.v_k(D, k)) for k in range(1, D)]
    W = [mk(wl.w_k(D, k)) for k in range(1, D)]
    ctA = encr.encrypt(enc.encode(A.reshape(-1), SCALE))
    ctB = encr.encrypt(enc.encode(B.reshape(-1), SCALE))

    ex = CountingExchange(par)
    run = lambda: par.sharded_cc_matrix_multiplication(ev, ctA, ctB, D, sigma, tau, V, W, keys, plans, rank, world, ex)
    for _ in range(args.warmup):
        out = run()
    torch.cuda.synchronize()
    ex.sent = ex.received = 0
    times = []
    for _ in range(args.reps):
        dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = run()
        torch.cuda.synchronize()
        t = torch.tensor([(time.perf_counter() - t0) * 1e3], device=ctx.device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)            # a product is done when its slowest rank is
        times.append(float(t.item()))
    sent, received = ex.sent // args.reps, ex.received // args.reps
    mem_peak = torch.cuda.max_memory_allocated(ctx.device)
    counts = torch.tensor([sent, received, mem_peak], device=ctx.device, dtype=torch.int64)
    allc = [torch.zeros_like(counts) for _ in range(world)]
    dist.all_gather(allc, counts)

    dd = D * D
    shards = [par.shard_rotations_shared(list(range(dd)), q, world) for q in range(world)]
    own = len(par.owned_block(D - 1, rank, world))
    bw = grouped_bandwidth(eng, ctx, ev, world, own, ctA.limbs) if own else None

    if rank == 0:
        unsharded = []
        for i in range(args.warmup + args.reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            want = wl.cc_matrix_multiplication_sparse(ev, ctA, ctB, D, sigma, tau, V, W, keys, plans)
            torch.cuda.synchronize()
            if i >= args.warmup:
                unsharded.append((time.perf_counter() - t0) * 1e3)
        same = bool(out.limbs == want.limbs and out.scale == want.scale and
                    torch.equal(out.data[:, :, :out.limbs], want.data[:, :, :want.limbs]))
        got = enc.decode(client.Decryptor(ctx, kg.secret_key()).decrypt(out))[0, :dd].reshape(D, D)
        ks = [4 * (plans.get(s).keyswitches_shared + 1) for s in shards]
        res = {
            "workload": "CC_Matrix_Multiplication d=%d, N=16384, {60,40,40,40,40,60}, power-of-two Galois keys, "
                        "d^2 rotations per transform sharded over %d GPU(s)" % (D, world),
            "gpus": world, "gpu": gpu_info(local),
            "ms_per_product": float(np.median(times)), "ms_min": min(times), "ms_max": max(times), "ms_all": times,
            "timing": "host clock around one product ended by a device synchronise on every rank, slowest rank, "
                      "%d repetitions after %d warm-up" % (args.reps, args.warmup),
            "products_per_s": 1e3 / float(np.median(times)),
            "ms_unsharded_one_gpu": float(np.median(unsharded)), "ms_unsharded_all": unsharded,
            "key_switches_per_gpu": ks, "key_switches_one_gpu": 4 * (plans.get(range(dd)).keyswitches_shared + 1),
            "rotations_per_gpu": [len(s) for s in shards],
            "products_owned_per_gpu": [len(par.owned_block(D - 1, q, world)) for q in range(world)],
            "bytes_sent_per_rank": [int(c[0]) for c in allc], "bytes_received_per_rank": [int(c[1]) for c in allc],
            "peak_device_memory_bytes_per_rank": [int(c[2]) for c in allc],
            "add_many_grouped_rank0": bw,
            "bit_identical_to_unsharded": same,
            "max_abs_err_vs_plain_AB": float(np.abs(got - A @ B).max()),
        }
        os.makedirs(args.out_dir, exist_ok=True)
        path = os.path.join(args.out_dir, "r03_matmul_scaling_%dgpu.json" % world)
        json.dump(res, open(path, "w"), indent=1)
        print(json.dumps({k: res[k] for k in ("gpus", "ms_per_product", "ms_min", "ms_max", "ms_unsharded_one_gpu",
                                              "bit_identical_to_unsharded",
                                              "max_abs_err_vs_plain_AB", "key_switches_per_gpu")}), flush=True)
        print("wrote", path, flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
