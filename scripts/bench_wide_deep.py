#!/usr/bin/env python
"""bench_wide_deep.py - BASELINE config 4 (wide+deep: 500 dense + 5000 one-hot columns = 50 categorical columns x 100 values,
MLP [1024, 512] relu, momentum, bf16) trained on N B200s, batch 8192 rows per GPU, 32 resident batches per rank.

    python scripts/bench_wide_deep.py --out DIR [--steps K] [--warmup W]
    python -m torch.distributed.run --nproc-per-node N scripts/bench_wide_deep.py --out DIR [--single-gpu DIR1/wide_deep.json]

Legs (one JSON, DIR/wide_deep.json, also printed):
  resident_sparse  sb_trainer_load_dataset_sparse + sb_trainer_run_resident: dense block as bf16 in HBM read by TMA, index rows
                   read through the step descriptor, four steps per captured graph
  dense_onehot     the same net, init and batches as a dense net on the materialised one-hot matrix (load_dataset + run_resident)
  host_fed_sparse  sb_trainer_step_sparse on pageable host batches (what the worker ran before the resident path)
  kernels          sb_trainer_profile_step of one sparse step: per-launch device time (embed_gather / embed_scatter share)
  parity           legs 1 and 2 run the same K steps from the same init: max |d theta| and max |d loss| of the loss curves
Timing follows bench.py: every captured graph warmed up, CUDA events on the trainer's stream with barrier + sync on both
sides, max over ranks; a timed region that did not run exactly --steps steps is an error.  The resident sets (310 MB sparse,
2.9 GB one-hot per rank) are larger than the 126 MB L2."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SEED = 20261017
N_DENSE, VOCAB, HIDDEN, BATCH, N_BATCHES, LR = 500, [100] * 50, [1024, 512], 8192, 32, 0.01
BF16_LOSS_TOL = 1e-4        # per-step bound of the resident bf16 loss curve at momentum (tests/test_benchmarked_paths.py, cfg2)


def work_per_row(n_dense, vocab, hidden):
    """algorithmic work per training row, by the rule of bench.flops_per_row (F_train = 6 sum(W) - 2 W_1, no dA for layer 0),
    and the resident bytes per row (bf16 operand rows at their 8-element pitch, int32 indices, fp32 y and w)"""
    n_onehot, n_cat = int(sum(vocab)), len(vocab)

    def f_train(f_in):
        dims = [f_in] + list(hidden) + [1]
        sw = sum(a * b for a, b in zip(dims[:-1], dims[1:]))
        return 6 * sw - 2 * dims[0] * dims[1]

    pitch = lambda n: (n + 7) // 8 * 8
    return {"sparse": {"gemm_flop": f_train(n_dense), "embed_adds": 2 * n_cat * hidden[0],
                       "bytes": 2 * pitch(n_dense) + 4 * n_cat + 8},
            "dense_onehot": {"gemm_flop": f_train(n_dense + n_onehot), "bytes": 2 * pitch(n_dense + n_onehot) + 8}}


def synth(rank, rows):
    """dense block ~ N(0, 1) clipped to +-4, one Zipf-distributed value per categorical column (5 % missing), y ~ Bernoulli(0.2),
    w = 1; seeded per rank"""
    rng = np.random.default_rng(SEED + 1000 * rank)
    Xd = np.clip(rng.standard_normal((rows, N_DENSE), dtype=np.float32), -4, 4)
    offs = np.concatenate([[0], np.cumsum(VOCAB)[:-1]])
    idx = np.empty((rows, len(VOCAB)), np.int32)
    for c, (V, o) in enumerate(zip(VOCAB, offs)):
        p = 1.0 / np.arange(1, V + 1); p /= p.sum()
        idx[:, c] = o + rng.choice(V, size=rows, p=p)
    idx[rng.random(idx.shape) < 0.05] = -1
    y = (rng.random(rows, dtype=np.float32) < 0.2).astype(np.float32)
    return Xd, idx, y, np.ones(rows, np.float32)


def onehot(Xd, idx, n_onehot):
    X = np.zeros((len(Xd), Xd.shape[1] + n_onehot), np.float32)
    X[:, :Xd.shape[1]] = Xd
    r = np.repeat(np.arange(len(idx)), idx.shape[1])
    j = idx.reshape(-1)
    X[r[j >= 0], Xd.shape[1] + j[j >= 0]] = 1.0       # (the categorical columns own disjoint column ranges)
    return X


def card(local_rank):
    """name and power limit of this GPU, read now (a query only)"""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(local_rank)],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:          # the numbers are still reported, marked as measured on an unnamed card
        return {"name": None, "power_limit": None, "error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--host-steps", type=int, default=50)
    ap.add_argument("--parity-steps", type=int, default=0, help="steps of the parity leg (default: --steps)")
    ap.add_argument("--single-gpu", default=None, help="wide_deep.json of an N = 1 run: weak-scaling efficiency against it")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    import torch
    import torch.distributed as dist
    import shifu_tensorflow_b200 as sb
    from shifu_tensorflow_b200 import dist_util

    if sb.capi.device_count() < 1:
        raise RuntimeError("bench_wide_deep.py needs a B200")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if world == 1:
            return v
        tns = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(tns, op=dist.ReduceOp.MAX)
        return float(tns.item())

    B, nb, n_onehot = BATCH, N_BATCHES, int(sum(VOCAB))
    F = N_DENSE + n_onehot
    K = args.steps
    Kp = args.parity_steps or K
    Xd, idx, y, w = synth(rank, nb * B)

    def make(sparse):
        uid = None
        if world > 1:
            uid = dist_util.broadcast_bytes(dist, sb.capi.nccl_unique_id, sb.capi.SB_NCCL_ID_BYTES, rank, device="cuda")
        desc = sb.make_desc(F, HIDDEN, [sb.ACT_RELU] * len(HIDDEN), loss=sb.LOSS_MSE, optimizer=sb.OPT_MOMENTUM, learning_rate=LR,
                            max_batch=B, precision=sb.PREC_BF16)
        t = sb.Trainer(desc, device=local_rank, nccl_id=uid, rank=rank, world=world)
        if world > 1 and os.environ.get("SB_EXCHANGE", "p2p") == "p2p":
            dist_util.enable_peer_exchange(dist, t, world, device="cuda")
        t.init_xavier(SEED)
        if sparse:
            t.set_sparse(N_DENSE, n_onehot, len(VOCAB))
        return t

    ts = make(True)
    ts.load_dataset_sparse(Xd, idx, y, w)
    td = make(False)
    td.load_dataset(onehot(Xd, idx, n_onehot), y, w)
    offsets = lambda first, n: [((first + i) % nb) * B for i in range(n)]

    # ---- parity at the timed size: the same Kp steps from the same init through both forms ----
    for t in (ts, td):
        t.run_resident(offsets(0, Kp), B)
    hist_s, hist_d = ts.loss_history(1, Kp), td.loss_history(1, Kp)
    th_s, th_d = ts.get_params(), td.get_params()
    barrier()
    dloss = float(np.abs(hist_s - hist_d).max())
    parity = {"steps": Kp, "max_abs_dtheta": float(np.abs(th_s - th_d).max()), "max_abs_dloss": dloss,
              "loss_first_last": [float(hist_s[0]), float(hist_s[-1])], "loss_tolerance": BF16_LOSS_TOL,
              "within_tolerance": bool(dloss <= BF16_LOSS_TOL)}

    def timed_resident(t):
        """bench.py's protocol: both multi-step graphs and the two single-step graphs warmed up, then K steps in one call"""
        stream = torch.cuda.ExternalStream(t.stream, device=torch.device("cuda", local_rank))
        t.run_resident(offsets(0, max(args.warmup, 8)), B)
        for i in range(2):
            t.step_resident_async(i * B, B)
        t.sync()
        barrier()
        step0 = t.global_step
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record(stream)
        t.run_resident(offsets(args.warmup, K), B)
        ev1.record(stream)
        t.sync()
        barrier()
        if t.global_step - step0 != K:
            raise RuntimeError("timed %d steps, --steps asked for %d" % (t.global_step - step0, K))
        ms = max_over_ranks(ev0.elapsed_time(ev1))
        return {"value": world * B * K / (ms / 1e3), "unit": "rows/s", "ms_per_step": ms / K, "steps": K,
                "last_loss": t.last_loss()}

    res_sparse = timed_resident(ts)
    res_dense = timed_resident(td)
    td.close()

    # ---- host-fed sparse steps (pageable host batches; each call copies, checks the indices and waits for the loss) ----
    for i in range(3):
        o = i * B
        ts.step_sparse(Xd[o:o + B], idx[o:o + B], y[o:o + B], w[o:o + B])
    barrier()
    h0 = time.perf_counter()
    for i in range(args.host_steps):
        o = (i % nb) * B
        ts.step_sparse(Xd[o:o + B], idx[o:o + B], y[o:o + B], w[o:o + B])
    barrier()
    host_s = max_over_ranks(time.perf_counter() - h0)
    res_host = {"value": world * B * args.host_steps / host_s, "unit": "rows/s", "ms_per_step": 1e3 * host_s / args.host_steps,
                "steps": args.host_steps, "timer": "host wall clock around sb_trainer_step_sparse x steps (synchronous), max over ranks"}

    # ---- per-kernel device times of one sparse step (a separate, un-captured step with an event after every launch) ----
    ts.profile_step(0, B)
    prof = ts.profile_step(B, B)
    total = sum(ms for _, ms in prof)
    kernels = {}
    for nm, ms in prof:
        kernels[nm] = kernels.get(nm, 0.0) + ms
    barrier()
    ts.close()

    cnt = work_per_row(N_DENSE, VOCAB, HIDDEN)
    for leg, form in ((res_sparse, "sparse"), (res_dense, "dense_onehot"), (res_host, "sparse")):
        leg["tflops_per_gpu"] = leg["value"] / world * cnt[form]["gemm_flop"] / 1e12
    out = {"workload": "BASELINE config 4: %d dense + %d one-hot (%d x %d) cols, MLP %s relu, momentum lr %g, MSE-on-sigmoid, bf16, "
                       "%d rows/GPU/step, %d resident batches per rank" % (N_DENSE, n_onehot, len(VOCAB), VOCAB[0], HIDDEN, LR, B, nb),
           "n_gpus": world, "card": card(local_rank), "resident_sparse": res_sparse, "dense_onehot": res_dense,
           "host_fed_sparse": res_host, "speedup_resident_sparse_vs_dense_onehot": res_sparse["value"] / res_dense["value"],
           "speedup_resident_sparse_vs_host_fed": res_sparse["value"] / res_host["value"],
           "kernels": {"step_ms": total, "ms": kernels, "embed_share": (kernels.get("embed_gather", 0.0) + kernels.get("embed_scatter", 0.0)) / total,
                       "method": "sb_trainer_profile_step: one un-captured step, CUDA event after every launch (rank 0)"},
           "parity": parity, "work_per_row": cnt,
           "resident_bytes_per_rank": {"sparse": nb * B * cnt["sparse"]["bytes"], "dense_onehot": nb * B * cnt["dense_onehot"]["bytes"]}}
    if args.single_gpu:
        one = json.load(open(args.single_gpu))
        out["weak_scaling_efficiency"] = {leg: out[leg]["value"] / (world * one[leg]["value"]) for leg in ("resident_sparse", "dense_onehot")}
    if rank == 0:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "wide_deep.json"), "w") as f:
            json.dump(out, f, indent=1)
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()
    if not parity["within_tolerance"]:
        raise SystemExit("parity leg outside tolerance: max |d loss| = %.3g > %.1g" % (dloss, BF16_LOSS_TOL))


if __name__ == "__main__":
    main()
