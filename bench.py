#!/usr/bin/env python
"""bench.py - rows/sec of the tabular-DNN train step (BASELINE.json metric) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config cfg2|cfg1|cfg0] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
           bench.py --gpus N --steps K --warmup W

One "step" = one pass of the hot path over one mini-batch: load -> forward -> loss -> backward -> gradient mean over
ranks (peer-memory exchange kernels, NCCL as fallback) -> optimizer update.  The headline config is cfg2 (2000 cols x
8192 rows per GPU, MLP [1024,512,256], SGD+momentum) - the config BASELINE.json states both numeric targets on; cfg1 is
reported under `also`.

  value      K steps whose mini-batches are already resident in HBM (sb_trainer_run_resident = the per-epoch batch loop in
             one call), CUDA events on the trainer's stream, barrier + sync on both sides, max over ranks (burst: ~30 ms)
  sustained  the same call for >= 3 s (clocks settle under the power cap); divided by the SUSTAINED measured peak
  e2e        the same step through the public C-ABI call with HOST (pinned) buffers: H2D of every batch and the read-back
             of the loss scalars inside the timed region
  roofline   per-kernel spans measured INSIDE the captured step graph (%globaltimer stamps of every kernel, slot "deps
             resolved" .. "last CTA exit"), so that the kernel times are the in-step times and sum to <= ms_per_step
  eval       BASELINE config 5: batch scoring of the trained 2000-col net, device-resident 100 M rows and host-buffer e2e
  cpu_baseline / --impl reference   the reference-equivalent CPU worker (oracle port on torch-CPU) on the host cores

Weak scaling: every rank owns its own `batch` rows per step.  PyTorch is plumbing only (rendezvous, barrier, max-reduce,
events, synthetic device data for the eval leg); all compute is libshifu_b200.so.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED = 20260921
# BASELINE.json configs.  Activation: relu (ModelConfig ActivationFunc); loss: the reference's MSE-on-sigmoid
# (res/ssgd_monitor.py:129) - same cost as the sigmoid-CE variant.
CONFIGS = {
    "cfg0": dict(F=200, hidden=[100, 50], batch=100, optimizer="adadelta", lr=1.0, n_batches=90),
    "cfg1": dict(F=1000, hidden=[512, 256, 128], batch=4096, optimizer="adam", lr=0.001, n_batches=64),
    "cfg2": dict(F=2000, hidden=[1024, 512, 256], batch=8192, optimizer="momentum", lr=0.01, n_batches=32),
}
OPT_ID = {"adadelta": 0, "adam": 1, "sgd": 2, "momentum": 3}
EVAL_ROWS = 100_000_000          # BASELINE config 5
EVAL_CHUNK = 1 << 20             # rows generated on the device per chunk (8.4 GB fp32 at 2000 cols)


def flops_per_row(F, hidden):
    """BASELINE.md section 3: F_train = 6*sum(W) - 2*W_1; hidden-GEMM share drops the out=1 layer (6*h_L)."""
    dims = [F] + list(hidden) + [1]
    sw = sum(a * b for a, b in zip(dims[:-1], dims[1:]))
    f_train = 6 * sw - 2 * dims[0] * dims[1]
    return f_train, f_train - 6 * hidden[-1], 2 * sw


def synth_dataset(cfg, rank, n_batches=None):
    """X~N(0,1) clipped +-4 fp32 row-major, y~Bernoulli(0.2), w=1 (BASELINE.md section 4); per-rank seed."""
    nb = n_batches or cfg["n_batches"]
    rows = nb * cfg["batch"]
    rng = np.random.default_rng(SEED + 1000 * rank)
    X = rng.standard_normal((rows, cfg["F"]), dtype=np.float32)
    np.clip(X, -4, 4, out=X)
    y = (rng.random(rows, dtype=np.float32) < 0.2).astype(np.float32)
    w = np.ones(rows, np.float32)
    return X, y, w


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index, period_ms=50):
        self.gpu, self.lines, self.proc, self.period = gpu_index, [], None, period_ms

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms",
                                          str(self.period), "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def window(self, t0, t1):
        """summary of the samples taken in [t0, t1] (perf_counter seconds); the sampler keeps running"""
        if not self.proc:
            return None
        sm, mx, pw, reasons = [], [], [], set()
        for ts, line in list(self.lines):
            if not (t0 - 0.06 <= ts <= t1 + 0.12):
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except Exception:
                continue
            for nm, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "power_w_max": float(max(pw)),
                "reasons": sorted(reasons), "samples": len(sm)}

    def stop(self):
        if self.proc:
            time.sleep(0.12)
            self.proc.terminate()


def host_threads() -> int:
    """threads the CPU arm may really use: affinity mask and cgroup quota, not the box's core count"""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(p))))
    except Exception:
        pass
    return n


def config_block(name, cfg, world):
    return {"workload": "%s: %d cols x %d rows/GPU/step, MLP %s relu, %s, MSE-on-sigmoid loss" %
                        (name, cfg["F"], cfg["batch"], cfg["hidden"], cfg["optimizer"]),
            "global_batch": cfg["batch"] * world, "rows_per_gpu": cfg["batch"], "parallelism": "dp%d" % world,
            "resident_set": "%d batches (%.0f MB fp32 per GPU) cycled, larger than the 126 MB L2 (no L2 flush needed)" %
                            (cfg["n_batches"], cfg["n_batches"] * cfg["batch"] * cfg["F"] * 4 / 1e6)}


def time_cpu_worker(cfg, name, min_seconds, warm_seconds, threads):
    """The reference-equivalent CPU worker (oracle/torch_cpu_worker.py: the ssgd_monitor.py batch loop on torch-CPU fp32)
    with ONE warm policy for both CPU numbers of this file: warm up for `warm_seconds` (thread pools, allocator, caches),
    then time whole passes over 4 mini-batches until `min_seconds` have elapsed."""
    import torch
    from oracle import shifu_oracle as so
    from oracle.torch_cpu_worker import TorchCpuWorker
    torch.set_num_threads(threads)
    net = so.NetDesc(cfg["F"], cfg["hidden"], [so.ACT_RELU] * len(cfg["hidden"]))
    params = so.xavier_init(net, SEED % 100000)
    opt = so.OptConfig(kind=OPT_ID[cfg["optimizer"]], lr=cfg["lr"])
    nb = min(4, cfg["n_batches"])
    X, y, w = synth_dataset(cfg, 0, nb)
    B = cfg["batch"]
    tb = [(torch.from_numpy(X[i * B:(i + 1) * B]), torch.from_numpy(y[i * B:(i + 1) * B].reshape(-1, 1)),
           torch.from_numpy(w[i * B:(i + 1) * B].reshape(-1, 1))) for i in range(nb)]
    wk = TorchCpuWorker(net, params, opt)
    t0, i = time.perf_counter(), 0
    while time.perf_counter() - t0 < warm_seconds or i < 3:
        wk.step(*tb[i % nb]); i += 1
    warm_steps = i
    t0, steps = time.perf_counter(), 0
    while True:
        wk.step(*tb[steps % nb]); steps += 1
        el = time.perf_counter() - t0
        if el >= min_seconds and steps >= 3:
            break
    return {"rows_per_sec": steps * B / el, "steps": steps, "seconds": el, "warm_steps": warm_steps, "cores": threads,
            "ms_per_step": 1e3 * el / steps}


def run_reference(args, cfg, rank, world):
    """`--impl reference`: the reference-equivalent CPU worker on the same config / metric.  TF 1.x + Python 2 cannot be
    installed here, so the oracle port IS the CPU arm (kind "port").  Under torchrun only rank 0 works.  `--warmup W` and
    `--steps K` are lower bounds: the warm-up also lasts >= 3 s and the timed region >= 5 s, the same policy as the
    `cpu_baseline` block of the b200 arm, so the two CPU numbers agree."""
    if rank != 0:
        return
    threads = host_threads()
    r = time_cpu_worker(cfg, args.config, min_seconds=5.0, warm_seconds=3.0, threads=threads)
    val = r["rows_per_sec"]
    out = {
        "impl": "reference", "metric": "rows/sec tabular-DNN train", "value": val, "unit": "rows/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "timed_steps": r["steps"], "warm_steps": r["warm_steps"],
        "ms_per_step": r["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_block(args.config, cfg, 1),
        "cpu_baseline": {"value": val, "unit": "rows/s", "cores": threads, "kind": "port",
                         "sample": "%d steps (%.1f s, after %d warm-up steps / 3 s) of %s (batch %d) on torch-CPU fp32, batch loop only" %
                                   (r["steps"], r["seconds"], r["warm_steps"], args.config, cfg["batch"])},
        "e2e": {"value": val, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out), flush=True)


def step_timeline(names, stamps, B, F, hidden):
    """stamps [k,16] ns of the traced step: slot 0 entry (CTA 0), 2 dependencies resolved, 10 last CTA exit.  Names come from
    the library as role[layer][.chunk][@MxNxK] (Net::next_trace)."""
    L = len(hidden)
    rows = []
    for nm, st in zip(names, stamps):
        begin = int(st[2]) if st[2] else int(st[0])
        end = int(st[10])
        if not begin or not end:
            continue
        role, flops = nm, 0
        if "@" in nm:
            role, dims = nm.split("@")
            M, N, K = (int(v) for v in dims.split("x"))
            flops = 2 * M * N * K
            if role.startswith("fwd_out"):
                role = "fwd%s+out" % role[len("fwd_out"):]
        cta0 = None
        if flops and st[3] and st[6]:      # CTA 0's pipeline milestones (us after its dependencies resolved)
            cta0 = {"first_tma": (int(st[3]) - begin) / 1e3, "first_acc": (int(st[6]) - begin) / 1e3,
                    "first_epilogue": (int(st[7]) - begin) / 1e3 if st[7] else None, "exit": (int(st[8]) - begin) / 1e3 if st[8] else None}
        elif role.startswith("xchg") and st[3]:
            # exchange kernel: every peer arrived (block 0) / last block's runs done / its stores fenced / every peer done
            cta0 = {"peers_arrived": (int(st[3]) - begin) / 1e3, "runs_done": (int(st[4]) - begin) / 1e3 if st[4] else None,
                    "fenced": (int(st[5]) - begin) / 1e3 if st[5] else None, "peers_done": (int(st[6]) - begin) / 1e3 if st[6] else None}
        rows.append({"kernel": role, "entry": int(st[0]), "begin": begin, "end": end, "flops": flops, "cta0": cta0})
    if not rows:
        return None
    t0 = min(r["begin"] for r in rows)
    for r in rows:
        r["us"] = (r["end"] - r["begin"]) / 1e3
        r["begin_us"] = (r["begin"] - t0) / 1e3
        r["end_us"] = (r["end"] - t0) / 1e3
        r["tflops"] = (r["flops"] / (r["us"] * 1e-6) / 1e12) if r["flops"] and r["us"] > 0 else None
        del r["entry"], r["begin"], r["end"]
    span = max(r["end_us"] for r in rows)
    # union of the busy intervals (kernels of the two streams overlap)
    iv = sorted((r["begin_us"], r["end_us"]) for r in rows)
    busy, cur0, cur1 = 0.0, iv[0][0], iv[0][1]
    for a, b in iv[1:]:
        if a > cur1:
            busy += cur1 - cur0; cur0, cur1 = a, b
        else:
            cur1 = max(cur1, b)
    busy += cur1 - cur0
    return {"kernels": rows, "span_us": span, "busy_us": busy, "idle_us": span - busy}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--config", default="cfg2", choices=sorted(CONFIGS))
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eval", action="store_true", help="skip the batch-scoring leg (BASELINE config 5)")
    ap.add_argument("--no-sustained", action="store_true")
    ap.add_argument("--no-ingest", action="store_true", help="skip the text-ingest leg (load_data on the GPU)")
    ap.add_argument("--sustained-seconds", type=float, default=3.0)
    ap.add_argument("--e2e-steps", type=int, default=0, help="steps of the host-buffer leg (default: min(steps, 50))")
    ap.add_argument("--also", default="cfg1", help="second config measured on the resident leg only and reported under 'also' ('' = none)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of --config computed (its loss, the parameters it left) as DIR/*.npy")
    args = ap.parse_args()
    cfg = CONFIGS[args.config]
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, cfg, rank, world)
        return

    import torch
    import torch.distributed as dist
    import shifu_tensorflow_b200 as sb

    torch.cuda.set_device(local_rank)
    from shifu_tensorflow_b200 import dist_util
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

    prec = sb.PREC_BF16 if args.precision == "bf16" else sb.PREC_FP32
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_tf = float(peaks.get("bf16_tflops", 1590.0))
    peak_sus = float(peaks.get("bf16_tflops_sustained", 1400.0))
    peak_src = "measured burst (MEASURED_PEAKS.json bf16_tflops)" if peaks else "fallback 1.59 PF (B200_PROFILING.md)"
    # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` capture of this command
    # (scripts/summarize_ncu.py writes the file); null when no capture of the current build has been committed
    traffic_db = {}
    try:
        traffic_db = json.load(open(os.path.join(ROOT, "profiles", "ncu_r02_traffic.json")))
    except Exception:
        pass

    sampler = ClockSampler(local_rank).start() if rank == 0 else None

    def make_trainer(name, nb, trace=False):
        c = CONFIGS[name]
        B, F, hidden = c["batch"], c["F"], c["hidden"]
        uid = None
        if world > 1:
            uid = dist_util.broadcast_bytes(dist, sb.capi.nccl_unique_id, sb.capi.SB_NCCL_ID_BYTES, rank, device="cuda")
        desc = sb.make_desc(F, hidden, [sb.ACT_RELU] * len(hidden), loss=sb.LOSS_MSE, optimizer=OPT_ID[c["optimizer"]],
                            learning_rate=c["lr"], max_batch=B, precision=prec)
        if trace:
            os.environ["SB_STEP_TRACE"] = "1"
        try:
            t = sb.Trainer(desc, device=local_rank, nccl_id=uid, rank=rank, world=world)
        finally:
            os.environ.pop("SB_STEP_TRACE", None)
        exchange = "none"
        if world > 1:
            exchange = "nccl"
            if os.environ.get("SB_EXCHANGE", "p2p") == "p2p":
                dist_util.enable_peer_exchange(dist, t, world, device="cuda")
                exchange = "p2p (peer-memory exchange kernels over CUDA-IPC)"
        t.init_xavier(SEED)  # same seed on every rank -> identical replicas
        return t, exchange

    def measure(name, full):
        c = CONFIGS[name]
        B, F, hidden = c["batch"], c["F"], c["hidden"]
        nb = c["n_batches"] if full else min(c["n_batches"], 16)
        t, exchange = make_trainer(name, nb)
        X, y, w = synth_dataset(c, rank, nb)
        t.load_dataset(X, y, w)
        stream = torch.cuda.ExternalStream(t.stream, device=torch.device("cuda", local_rank))
        f_train, f_gemm, _ = flops_per_row(F, hidden)

        def timed_run(n_steps, first):
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            wall0 = time.perf_counter()
            ev0.record(stream)
            t.run_resident([((first + i) % nb) * B for i in range(n_steps)], B)
            ev1.record(stream)
            t.sync()
            barrier()
            wall1 = time.perf_counter()
            return max_over_ranks(ev0.elapsed_time(ev1)), wall0, wall1

        # ---------------- device-resident leg (value) ----------------
        # the per-epoch batch loop as ONE call (sb_trainer_run_resident: four steps per captured graph); at least two
        # chunks of four steps so that both captured multi-step graphs exist before the timed region, plus the two
        # single-step graphs a step count that is not a multiple of four ends with
        t.run_resident([(i % nb) * B for i in range(max(args.warmup, 8))], B)
        for i in range(2):
            t.step_resident_async((i % nb) * B, B)
        t.sync()
        barrier()
        time.sleep(0.3 if full else 0.0)
        step0 = t.global_step
        ms, wall0, wall1 = timed_run(args.steps, args.warmup)
        if t.global_step - step0 != args.steps:
            raise RuntimeError("timed %d steps, --steps asked for %d" % (t.global_step - step0, args.steps))
        clk = sampler.window(wall0, wall1) if (sampler and full) else None
        last_loss = t.last_loss()
        if full and args.dump_outputs:
            dump_outputs(args.dump_outputs, t, rank, barrier)
        value = world * B * args.steps / (ms / 1e3)
        res = {"value": value, "ms_per_step": ms / args.steps, "last_loss": last_loss, "clocks": clk,
               "gradient_exchange": exchange, "gpu_launches": t.kernels_per_step(B) * args.steps,
               "step_api": "sb_trainer_run_resident (one call for all steps, four steps per captured graph)",
               "config": config_block(name, dict(c, n_batches=nb), world)}

        # ---------------- sustained leg: the same call for >= 3 s ----------------
        if full and not args.no_sustained:
            n_sus = int(math.ceil(args.sustained_seconds * 1e3 / (ms / args.steps) / 4.0)) * 4
            ms_s, w0, w1 = timed_run(n_sus, 0)
            res["sustained"] = {"value": world * B * n_sus / (ms_s / 1e3), "unit": "rows/s", "steps": n_sus, "seconds": ms_s / 1e3,
                                "ms_per_step": ms_s / n_sus, "clocks": sampler.window(w0 + 0.5, w1) if sampler else None,
                                "step_fraction_of_sustained_peak": (B * n_sus / (ms_s / 1e3) * f_train / 1e12) / peak_sus,
                                "peak": peak_sus, "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (4 s cuBLAS loop)"}

        # ---------------- roofline: in-graph kernel spans ----------------
        roofline = None
        if prec == sb.PREC_BF16:
            tt, _ = make_trainer(name, nb, trace=True)
            tt.load_dataset(X[:4 * B], y[:4 * B], w[:4 * B])
            tt.run_resident([(i % 4) * B for i in range(16)], B)
            tt.sync()
            barrier()
            names, stamps = tt.debug_step_trace()
            tl = step_timeline(names, stamps, B, F, hidden)
            barrier()
            tt.close()
            if tl:
                gem = [k for k in tl["kernels"] if k["flops"]]
                top = max(gem, key=lambda k: k["us"])
                sum_us = sum(k["us"] for k in gem)
                key = "%s/%s" % (name, top["kernel"])
                roofline = {"bound": "tensor", "achieved": top["tflops"], "peak": peak_tf, "unit": "TFLOP/s",
                            "frac": top["tflops"] / peak_tf, "traffic": traffic_db.get(key),
                            "traffic_source": "profiles/ncu_r02_traffic.json (ncu --set full capture of this command)" if key in traffic_db else None,
                            "kernel": "gemm_tc_kernel %s (tcgen05 + TMA), the longest GEMM of the step" % top["kernel"],
                            "flops_per_launch": top["flops"], "kernel_us": top["us"], "peak_source": peak_src,
                            "method": "%globaltimer stamps inside the captured step graph of a second, traced trainer: dependencies "
                                      "resolved (CTA 0) .. last CTA exit of every kernel; no profiler, no extra launches",
                            "all_gemms": {"flops": sum(k["flops"] for k in gem), "sum_kernel_us": sum_us,
                                          "tflops": sum(k["flops"] for k in gem) / (sum_us * 1e-6) / 1e12,
                                          "frac": sum(k["flops"] for k in gem) / (sum_us * 1e-6) / 1e12 / peak_tf},
                            "step_span_us": tl["span_us"], "step_busy_us": tl["busy_us"], "step_idle_us": tl["idle_us"],
                            "step_fraction_of_peak": (value / world * f_train / 1e12) / peak_tf,
                            "kernels": [{k2: (round(v, 3) if isinstance(v, float) else
                                              ({a_: (round(b_, 2) if b_ is not None else None) for a_, b_ in v.items()} if isinstance(v, dict) else v))
                                         for k2, v in k.items()} for k in tl["kernels"]]}
        if roofline is None:
            roofline = {"bound": "tensor", "achieved": value / world * f_train / 1e12, "peak": peak_tf, "unit": "TFLOP/s",
                        "frac": (value / world * f_train / 1e12) / peak_tf, "traffic": None, "peak_source": peak_src,
                        "kernel": "whole step (no in-graph trace in this precision mode)"}
        res["roofline"] = roofline
        if not full:
            barrier()
            t.close()
            return res

        # ---------------- end-to-end leg: host (pinned) buffers through sb_trainer_step ----------------
        e2e_steps = args.e2e_steps or min(args.steps, 50)
        n_pin = 4
        pin = []
        for i in range(n_pin):
            px = torch.empty((B, F), dtype=torch.float32).pin_memory()
            py = torch.empty(B, dtype=torch.float32).pin_memory()
            pw = torch.empty(B, dtype=torch.float32).pin_memory()
            px.numpy()[:] = X[i * B:(i + 1) * B]; py.numpy()[:] = y[i * B:(i + 1) * B]; pw.numpy()[:] = w[i * B:(i + 1) * B]
            pin.append((px.numpy(), py.numpy(), pw.numpy()))
        for i in range(3):
            t.step(*pin[i % n_pin])
        barrier()
        e0 = time.perf_counter()
        for i in range(e2e_steps):
            t.step(*pin[i % n_pin])  # synchronous: H2D batch, load/cast kernel, step, D2H loss, host sees the loss
        barrier()
        sync_s = max_over_ranks(time.perf_counter() - e0)
        # pipelined public call: every step still copies its own batch H2D and its loss scalars D2H inside the timed
        # region, but the copy of batch i+1 overlaps the compute of batch i; the host reads the loss after the last step
        for i in range(3):
            t.step_async(*pin[i % n_pin])
        t.sync()
        barrier()
        e0 = time.perf_counter()
        for i in range(e2e_steps):
            t.step_async(*pin[i % n_pin])
        loss_h = t.last_loss()
        barrier()
        e2e_s = max_over_ranks(time.perf_counter() - e0)
        res["e2e"] = {"value": world * B * e2e_steps / e2e_s, "unit": "rows/s", "h2d_bytes_per_step": B * (F + 2) * 4,
                      "d2h_bytes_per_step": 16, "steps": e2e_steps, "ms_per_step": 1e3 * e2e_s / e2e_steps,
                      "synchronous_value": world * B * e2e_steps / sync_s, "last_loss": loss_h,
                      "timer": "host wall clock around sb_trainer_step_async x steps + sb_trainer_last_loss (pinned host buffers, "
                               "H2D of every batch and D2H of every step's loss scalars inside), max over ranks; "
                               "synchronous_value = the same with sb_trainer_step (host waits for each loss)"}
        trained = t.get_params()      # (sharded update: pulls every run's fp32 master from its owner rank)
        barrier()                     # no rank may free its arena while a peer still reads it
        t.close()

        # ---------------- eval leg: BASELINE config 5 (batch scoring of the trained net) ----------------
        res["eval"] = None
        if not args.no_eval and prec == sb.PREC_BF16:
            res["eval"] = eval_leg(sb, torch, c, trained, X, world, rank, local_rank, barrier, max_over_ranks, peak_tf)

        # ---------------- ingest leg: load_data's per-cell float() loop on the GPU (SURVEY 8f rank 1) ----------------
        res["ingest"] = None
        if rank == 0 and world == 1 and not args.no_ingest:
            res["ingest"] = ingest_leg(sb, local_rank, float(peaks.get("hbm_gbs", 6650.0)))

        # ---------------- CPU baseline (rank 0, N = 1 only) ----------------
        res["cpu_baseline"] = None
        if rank == 0 and world == 1 and not args.no_cpu_baseline:
            r = time_cpu_worker(c, name, min_seconds=10.0, warm_seconds=3.0, threads=host_threads())
            res["cpu_baseline"] = {"value": r["rows_per_sec"], "unit": "rows/s", "cores": r["cores"], "kind": "port",
                                   "sample": "%d steps (%.1f s, after %d warm-up steps / 3 s) of %s on torch-CPU fp32 = "
                                             "reference-equivalent worker loop (TF-1.x absent)" % (r["steps"], r["seconds"], r["warm_steps"], name)}
        return res

    main_res = measure(args.config, True)
    second = None
    if args.also and args.also != args.config and args.also in CONFIGS:
        second = measure(args.also, False)
    if sampler:
        sampler.stop()

    if rank == 0:
        out = {
            "metric": "rows/sec tabular-DNN train", "value": main_res["value"], "unit": "rows/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": main_res["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16" if prec == sb.PREC_BF16 else "f32", "data": "synthetic",
            "config": main_res["config"], "clocks": main_res["clocks"], "e2e": main_res["e2e"],
            "gpu_launches": main_res["gpu_launches"], "roofline": main_res["roofline"], "cpu_baseline": main_res["cpu_baseline"],
            "sustained": main_res.get("sustained"), "eval": main_res.get("eval"), "ingest": main_res.get("ingest"),
            "last_loss": main_res["last_loss"], "gradient_exchange": main_res["gradient_exchange"],
        }
        if second is not None:
            out["also"] = {k: second[k] for k in ("value", "ms_per_step", "config", "roofline", "last_loss", "gpu_launches")}
            out["also"]["unit"] = "rows/s"
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir, t, rank, barrier):
    """What the timed steps hand a caller of sb_trainer_run_resident, taken right after them: the mini-batch loss of the
    last step (loss.npy, [1]) and the parameters it left (params.npy, the flat layout of sb_trainer_get_params; 10.9 MB
    at cfg2), both float32.  The inputs (synthetic rows, Xavier init) are seeded, so two builds can be compared file by
    file; compare with a tolerance, since the order of the step's reductions is not fixed and two runs of one build
    differ in the last bits (cfg2, 50 + 12 steps: 1.2e-5 max abs on the parameters, on a B200 at 1000 W).  Every rank
    reads the parameters (a sharded update keeps them on their owner ranks); rank 0 writes."""
    params = t.get_params()
    loss = t.loss_history(t.global_step, 1)
    barrier()
    if rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        np.save(os.path.join(out_dir, "loss.npy"), loss)
        np.save(os.path.join(out_dir, "params.npy"), params)


def ingest_leg(sb, device, hbm_gbs):
    """load_data (ssgd_monitor.py:348-454) on the GPU: '|'-delimited normalised text -> fp32 columns, result left on the device
    (sb_text_parse_device).  cfg0-shaped rows (target + 200 features), 40 000 lines.  HBM roofline: the three kernels read the
    text three times (newline count, line offsets, cells) and write X once."""
    rows, F = 40000, 200
    rng = np.random.default_rng(SEED)
    vals = np.clip(rng.standard_normal((rows, F)), -4, 4)
    ys = (rng.random(rows) < 0.2).astype(int)
    text = "\n".join("%d|" % ys[i] + "|".join("%.6f" % v for v in vals[i]) for i in range(rows)).encode() + b"\n"
    col_map = [sb.capi.COL_TARGET] + list(range(F))
    sb.capi.text_parse_device(text[:200000 + text[200000:].index(b"\n") + 1], col_map, F, device=device)     # warm-up
    best_k, best_w = None, None
    for _ in range(3):
        t0 = time.perf_counter()
        X, y, w, flags, _, kms = sb.capi.text_parse_device(text, col_map, F, device=device)
        wall = time.perf_counter() - t0
        for a in (X, y, w):
            a.free()
        if best_k is None or kms < best_k:
            best_k = kms
        if best_w is None or wall < best_w:
            best_w = wall
    alg = 3 * len(text) + 4 * rows * (F + 2)
    ach = alg / (best_k * 1e-3) / 1e9
    # the reference's own loop on the same bytes: per-cell float() in Python (bounded sample: 2 000 lines)
    sample = text.split(b"\n", 2000)[:2000]
    t0 = time.perf_counter()
    for line in sample:
        cols = line.decode().split("|")
        float(cols[0]); [float(c) for c in cols[1:]]
    py_s = time.perf_counter() - t0
    py_bytes = sum(len(l) + 1 for l in sample)
    return {"metric": "text ingest (load_data)", "rows": rows, "cols": F + 1, "text_bytes": len(text), "flagged_cells": len(flags),
            "kernel_ms": best_k, "roofline": {"bound": "hbm", "achieved": ach, "peak": hbm_gbs, "unit": "GB/s", "frac": ach / hbm_gbs,
                                              "algorithmic_bytes": alg, "note": "3 x text read + X/y/w written once, device time of the three kernels"},
            "e2e": {"value": len(text) / best_w / 1e9, "unit": "GB/s of text", "seconds": best_w,
                    "note": "sb_text_parse_device wall time incl. cudaMalloc, H2D of the text and the host-side line-count prefix"},
            "cpu_baseline": {"value": py_bytes / py_s / 1e9, "unit": "GB/s of text", "kind": "reference loop (split + float() per cell, "
                             "ssgd_monitor.py:387-410), 2 000 lines, 1 thread"}}


def eval_leg(sb, torch, c, trained_params, X_host, world, rank, local_rank, barrier, max_over_ranks, peak_tf):
    """BASELINE config 5 (TensorflowModel.compute, TensorflowModel.java:53-94, 100 M rows of the 2000-col net on one B200):
    rows are sharded over the ranks with no collective (strong scaling of the 100 M-row job).
      device-resident  synthetic fp32 rows generated on the device in 1 Mi-row chunks (8.4 GB, >> L2), scored with
                       sb_model_score_device (cast + forward GEMMs + output layer), CUDA events on the model's stream
      e2e              sb_model_score on pinned HOST rows: H2D of the features and D2H of the scores inside"""
    F, hidden = c["F"], c["hidden"]
    desc = sb.make_desc(F, hidden, [sb.ACT_RELU] * len(hidden), precision=sb.PREC_BF16)
    m = sb.Model.create(desc, trained_params, device=local_rank)
    dev = torch.device("cuda", local_rank)
    stream = torch.cuda.ExternalStream(m.stream, device=dev)
    my_rows = EVAL_ROWS // world
    chunk = min(EVAL_CHUNK, my_rows)
    g = torch.Generator(device=dev); g.manual_seed(SEED + rank)
    Xd = torch.empty((chunk, F), dtype=torch.float32, device=dev).normal_(generator=g).clamp_(-4, 4)
    out = torch.empty(chunk, dtype=torch.float32, device=dev)
    torch.cuda.synchronize()
    m.score_device(Xd.data_ptr(), chunk, out.data_ptr()); m.sync()          # warm-up (lazy module load)
    n_chunks = my_rows // chunk
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(stream)
    for _ in range(n_chunks):
        m.score_device(Xd.data_ptr(), chunk, out.data_ptr())
    ev1.record(stream)
    m.sync()
    barrier()
    ms = max_over_ranks(ev0.elapsed_time(ev1))
    rows_done = n_chunks * chunk * world
    _, _, f_score = flops_per_row(F, hidden)
    val = rows_done / (ms / 1e3)
    mean_score = float(out.mean().item())
    del Xd, out
    # end to end from pinned host rows
    n_host = min(len(X_host), 131072)
    px = torch.empty((n_host, F), dtype=torch.float32).pin_memory()
    px.numpy()[:] = X_host[:n_host]
    m.score(px.numpy()[:4096])
    barrier()
    e0 = time.perf_counter()
    sc = m.score(px.numpy())
    barrier()
    e2e_s = max_over_ranks(time.perf_counter() - e0)
    m.close()
    # the two tensor-core parity modes on the same net (device-resident, a shorter run): fp32-class scores, 6 / 3 part products
    parity = {}
    for pname, pid in (("fp32_tc", sb.PREC_FP32_TC), ("bf16x2", sb.PREC_BF16X2)):
        mp = sb.Model.create(sb.make_desc(F, hidden, [sb.ACT_RELU] * len(hidden), precision=pid), trained_params, device=local_rank)
        sp = torch.cuda.ExternalStream(mp.stream, device=dev)
        rows_p = 1 << 18
        Xp = torch.empty((rows_p, F), dtype=torch.float32, device=dev).normal_(generator=g).clamp_(-4, 4)
        op = torch.empty(rows_p, dtype=torch.float32, device=dev)
        torch.cuda.synchronize()
        mp.score_device(Xp.data_ptr(), rows_p, op.data_ptr()); mp.sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 8
        e0.record(sp)
        for _ in range(reps):
            mp.score_device(Xp.data_ptr(), rows_p, op.data_ptr())
        e1.record(sp)
        mp.sync()
        msp = e0.elapsed_time(e1)
        parity[pname] = {"value": reps * rows_p / (msp / 1e3), "unit": "rows/s", "rows": reps * rows_p,
                         "mma_products_per_contraction": 6 if pname == "fp32_tc" else 3}
        mp.close()
        del Xp, op
    return {"metric": "rows/sec batch scoring (eval path)", "value": val, "parity_modes": parity, "unit": "rows/s", "rows": rows_done, "seconds": ms / 1e3,
            "dtype": "bf16", "workload": "BASELINE config 5: %d M rows x %d cols through MLP %s, %d rank(s), device-resident fp32 rows "
                                         "(1 Mi-row chunks, larger than L2)" % (rows_done // 1_000_000, F, hidden, world),
            "roofline": {"bound": "tensor", "achieved": val / world * f_score / 1e12, "peak": peak_tf, "unit": "TFLOP/s",
                         "frac": (val / world * f_score / 1e12) / peak_tf,
                         "note": "whole scoring pass incl. the fp32->bf16 cast kernel (HBM-bound, 12 KB/row) and the output layer"},
            "mean_score": mean_score,
            "e2e": {"value": world * n_host / e2e_s, "unit": "rows/s", "rows": n_host * world, "h2d_bytes": n_host * F * 4,
                    "d2h_bytes": n_host * 4, "mean_score": float(np.mean(sc)),
                    "timer": "host wall clock around sb_model_score on pinned host rows (H2D + cast + forward + D2H)"}}


if __name__ == "__main__":
    main()
