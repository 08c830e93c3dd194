#!/usr/bin/env python
"""Benchmark of the BASELINE.json metric: Flow.log_prob samples/s on the 10-layer RQ-NSF, D=784, batch 2^20, sharded over N GPUs.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--rows R] [--weak] [--dump-outputs DIR]

One "step" = one Flow.log_prob pass over ONE synthetic Gaussian batch of R rows (default 2^20, BASELINE.json configs[2]).
With N GPUs (torchrun, one rank per GPU) the batch is SHARDED: every rank owns R/N rows and a replica of the weights
(strong scaling, BASELINE.md section 3.3); the only collective is the all-gather of the per-sample log-probs.  `--weak`
gives every rank R rows instead (the round-1 measurement).  Prints ONE JSON line (rank 0).  DESIGN.md section 6 explains
every key.
"""
import os
os.environ.setdefault("NCCL_DEBUG", "WARN")      # keep NCCL's version banner off stdout: rank 0 prints ONE JSON line
import argparse
import json
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

FEATURES, HIDDEN, LAYERS, BINS, BLOCKS = 784, 256, 10, 8, 2
METRIC = "Flow.log_prob samples/sec, 10-layer RQ-NSF D=784"
WORKLOAD = "cfg3 10x[ActNorm,RandPerm+LULinear,RQ-coupling(H=256,2 blocks,K=8,B=3)] D=784 log_prob"
# algorithmic work per sample (SURVEY.md section 8d)
D_ID = FEATURES // 2
M_PARAMS = 3 * BINS - 1
FLOP_COND_PER_ROW = 2 * (D_ID * HIDDEN + 2 * BLOCKS * HIDDEN * HIDDEN + HIDDEN * D_ID * M_PARAMS)   # one coupling's conditioner
FLOP_FINAL_PER_ROW = 2 * HIDDEN * (D_ID * M_PARAMS)                                                 # ... its final layer alone
FLOP_AFFINE_PER_ROW = 2 * FEATURES * FEATURES
FLOP_PER_SAMPLE = LAYERS * (FLOP_COND_PER_ROW + FLOP_AFFINE_PER_ROW)
#: MMA flops the coupling-step kernel executes per row: 3 fp16 MMAs per product; K = 392 padded to 13 slabs of 32; 24 packed
#: rows per 23-parameter feature
MMA_EXEC_STEP_PER_ROW = 3 * 2 * (416 * HIDDEN + 2 * BLOCKS * HIDDEN * HIDDEN + HIDDEN * D_ID * 24)
#: round-1 launch sequence (NFLOWS_B200_STEP_KERNEL=0): final layer in 240-column tiles, 24/23 rows per feature, 400/392 features
FUSED_PAD = (24.0 / 23.0) * (400.0 / 392.0)


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"], "bf16_tflops_sustained": p.get(
            "bf16_tflops_sustained", p["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        time.sleep(0.05)
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for name, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        smax = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def host_threads():
    """Threads for the CPU arm: the cores this process may run on (not the box's logical CPU count: 128 threads on a 64-core
    allowance ran the oracle 40x slower), capped at 64; NFLOWS_REF_THREADS overrides.  torchrun's OMP_NUM_THREADS=1 is undone."""
    env = os.environ.get("NFLOWS_REF_THREADS")
    if env:
        return max(1, int(env))
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    return max(1, min(64, n))


def build_flow(seed=0):
    from nflows_b200.flows import recipes
    torch.manual_seed(seed)
    return recipes.perturb_(recipes.rq_nsf(FEATURES, HIDDEN, LAYERS, num_bins=BINS, tail_bound=3.0, num_blocks=BLOCKS).eval())


def workload_config(args, world):
    """The `config` object of the JSON line -- the SAME keys for the native and the reference arm."""
    rows = args.rows if args.weak else args.rows // world
    return {"workload": WORKLOAD, "global_batch": rows * world, "rows_per_gpu": rows,
            "parallelism": "dp%d batch-shard, %s" % (world, "weak: %d rows per GPU" % rows if args.weak else "one 2^20-row batch sharded"),
            "l2": "inputs (%.1f GB/GPU) exceed the 126 MB L2; no flush needed" % (rows * FEATURES * 4 / 1e9)}


def cpu_oracle_rate(flow, budget_s=12.0, chunk=2048, max_rows=1 << 15):
    """The CPU restatement of the reference path (oracle/, torch ATen fp32, all host threads) on a bounded sample."""
    from oracle import flow_oracle as O
    sd = {k: v.detach().cpu().clone() for k, v in flow.state_dict().items()}
    spec = O.nsf_spec(LAYERS, num_bins=BINS, tail_bound=3.0)
    g = torch.Generator().manual_seed(123)
    x = torch.randn(chunk, FEATURES, generator=g)
    with torch.no_grad():
        O.flow_log_prob(sd, spec, x[:256])      # warm-up
        rows, t0 = 0, time.perf_counter()
        while rows < max_rows and time.perf_counter() - t0 < budget_s:
            O.flow_log_prob(sd, spec, x)
            rows += chunk
        dt = time.perf_counter() - t0
    return rows / dt, rows, torch.get_num_threads()


def torch_cuda_rate(flow, dev, budget_s=3.0, chunks=(1 << 14, 1 << 15, 1 << 16, 1 << 17)):
    """SURVEY.md section 8(d) "reference-CUDA baseline": the restatement of the reference path (oracle/, plain torch ops, true-fp32
    matmuls) with weights and data on the GPU, looped over chunks so the [chunk, d_t * 23] parameter tensor the reference
    materialises fits; the chunk size is swept and the best rate reported.  A context figure like cpu_baseline; none of this
    package's kernels run here."""
    from oracle import flow_oracle as O
    torch.backends.cuda.matmul.allow_tf32 = False
    sd = {k: v.detach().to(dev).clone() for k, v in flow.state_dict().items()}
    spec = O.nsf_spec(LAYERS, num_bins=BINS, tail_bound=3.0)
    g = torch.Generator(device=dev).manual_seed(123)
    best, tried = None, {}
    for chunk in chunks:
        try:
            x = torch.randn(chunk, FEATURES, device=dev, generator=g)
            with torch.no_grad():
                O.flow_log_prob(sd, spec, x)
                torch.cuda.synchronize()
                rows, t0 = 0, time.perf_counter()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                while rows < (1 << 19) and time.perf_counter() - t0 < budget_s:
                    O.flow_log_prob(sd, spec, x)
                    rows += chunk
                    torch.cuda.synchronize()
                e1.record()
                torch.cuda.synchronize()
            rate = rows / (e0.elapsed_time(e1) * 1e-3)
            tried[str(chunk)] = round(rate, 1)
            if best is None or rate > best[0]:
                best = (rate, chunk, rows)
            del x
        except RuntimeError as exc:           # out of memory at this chunk size: keep what fitted
            tried[str(chunk)] = "failed: %s" % str(exc).split("\n")[0][:80]
            torch.cuda.empty_cache()
            break
    return best, tried


def spline_hbm_roofline(dev, peaks, rows=1 << 20, d_t=32, bins=8, iters=10):
    """The HBM-bound spline segment (BASELINE configs[1] shape): conditioner output [rows, d_t*(3K-1)] resident in HBM ->
    nfk_rqs_rows.  Algorithmic bytes = 4*(M+2) per transformed element + 4 per identity element copied (read+write)."""
    from nflows_b200 import _native as N
    from nflows_b200 import kernels as K
    m = 3 * bins - 1
    g = torch.Generator(device=dev).manual_seed(7)
    x = torch.randn(rows, 2 * d_t, device=dev, generator=g)
    params = torch.randn(rows, d_t * m, device=dev, generator=g)
    t_cols = torch.arange(0, 2 * d_t, 2, device=dev, dtype=torch.int32)
    id_cols = torch.arange(1, 2 * d_t, 2, device=dev, dtype=torch.int32)
    lad = torch.zeros(rows, device=dev)
    y = torch.empty_like(x)
    flags = K.new_flags(dev)
    desc = N.spline_desc(bins, "linear", 3.0, 0, 1, 0, 1, 1e-3, 1e-3, 1e-3, False, 128.0 ** 0.5)
    for _ in range(3):
        K.rqs_rows(desc, False, x, params, t_cols, id_cols, lad, flags, out=y)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        K.rqs_rows(desc, False, x, params, t_cols, id_cols, lad, flags, out=y)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    nbytes = rows * (d_t * (4 * (m + 2)) + d_t * 8 + 8)
    achieved = nbytes / (ms * 1e-3) / 1e9
    return {"kernel": "rqs_rows_kernel<8,exact>", "bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
            "frac": achieved / peaks["hbm_gbs"], "traffic": None, "avg_launch_ms": ms,
            "workload": "rows=2^20 d_t=32 K=8 params in HBM (3.2 GB > L2)", "peak_kind": "copy bandwidth, %s" % peaks["source"]}


def extra_workloads(dev, flow):
    """The other single-GPU configurations of BASELINE.json, one short timing each (CUDA events, 3 warm-ups): cfg 2 (single RQ
    coupling D=64 forward + inverse at 2^20 rows), Flow.sample of the cfg-3 flow, cfg 4 (autoregressive RQ inverse, 2^18 x 64)."""
    from nflows_b200 import transforms as T
    from nflows_b200.flows import recipes
    out = {}

    def timed(fn, iters=5, warm=3):
        for _ in range(warm):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters

    with torch.no_grad():
        try:
            torch.manual_seed(0)
            layer = recipes.rq_coupling_layer(64, 128).eval().to(dev)
            x = torch.randn(1 << 20, 64, device=dev)
            y, _ = layer(x)
            ms_f = timed(lambda: layer(x))
            ms_i = timed(lambda: layer.inverse(y))
            out["cfg2_rq_coupling_D64_2^20"] = {"forward_ms": ms_f, "inverse_ms": ms_i,
                                                "forward_samples_per_s": (1 << 20) / (ms_f * 1e-3),
                                                "inverse_samples_per_s": (1 << 20) / (ms_i * 1e-3)}
            del x, y, layer
        except Exception as exc:
            out["cfg2_rq_coupling_D64_2^20"] = {"unavailable": "%s: %s" % (type(exc).__name__, exc)}
        try:
            n = 1 << 18
            ms = timed(lambda: flow.sample(n), iters=3, warm=2)
            out["cfg3_sample_2^18"] = {"ms": ms, "samples_per_s": n / (ms * 1e-3)}
        except Exception as exc:
            out["cfg3_sample_2^18"] = {"unavailable": "%s: %s" % (type(exc).__name__, exc)}
        try:
            torch.manual_seed(0)
            ar = T.MaskedPiecewiseRationalQuadraticAutoregressiveTransform(features=64, hidden_features=256, num_bins=8, tails="linear",
                                                                            tail_bound=3.0, num_blocks=2).eval().to(dev)
            z = torch.randn(1 << 18, 64, device=dev)
            ms = timed(lambda: ar.inverse(z), iters=2, warm=1)
            ms_f = timed(lambda: ar(z), iters=3, warm=2)
            out["cfg4_ar_rq_D64_2^18"] = {"inverse_ms": ms, "inverse_samples_per_s": (1 << 18) / (ms * 1e-3), "forward_ms": ms_f,
                                          "forward_samples_per_s": (1 << 18) / (ms_f * 1e-3)}
        except Exception as exc:
            out["cfg4_ar_rq_D64_2^18"] = {"unavailable": "%s: %s" % (type(exc).__name__, exc)}
        try:
            # cfg 5: Glow-style multiscale flow on 3x32x32 images (4 levels x 8 steps, 96 hidden channels), native pixel-row chain;
            # beside it the same flow as eager PyTorch (cuDNN convolutions) on this GPU, fp64 inputs never take the native path
            torch.manual_seed(0)
            glow = recipes.perturb_(recipes.glow_multiscale()).eval().to(dev)
            n = 512
            img = torch.randn(n, 3, 32, 32, device=dev)
            ms_lp = timed(lambda: glow.log_prob(img), iters=3, warm=2)
            ms_s = timed(lambda: glow.sample(n), iters=3, warm=2)
            rec = {"images": n, "log_prob_ms": ms_lp, "log_prob_images_per_s": n / (ms_lp * 1e-3), "sample_ms": ms_s,
                   "sample_images_per_s": n / (ms_s * 1e-3)}
            with torch.enable_grad():           # autograd on = the differentiable torch formulation of the same modules
                ms_eager = timed(lambda: glow.log_prob(img).detach(), iters=2, warm=1)
            rec["torch_eager_same_gpu_log_prob_ms"] = ms_eager
            want = glow.double().log_prob(img[:32].double()).float()
            got = glow.float().log_prob(img[:32])
            rec["log_prob_rel_err_vs_fp64"] = float(((got - want).abs() / torch.maximum(want.abs(), torch.ones_like(want))).max())
            out["cfg5_glow_3x32x32"] = rec
        except Exception as exc:
            out["cfg5_glow_3x32x32"] = {"unavailable": "%s: %s" % (type(exc).__name__, exc)}
    return out


def dump_outputs(directory, log_prob, limit_bytes=64 << 20):
    """Writes the per-sample log-probs as DIR/log_prob.npy (float32).  An output over `limit_bytes` is replaced by a fixed,
    seeded sample of rows, whose indices go to DIR/log_prob_rows.npy (float64, exact for any row count)."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    lp = log_prob.float().cpu()
    if lp.numel() * 4 > limit_bytes:
        rows = torch.randperm(lp.numel(), generator=torch.Generator().manual_seed(0))[:limit_bytes // 12].sort().values
        lp = lp[rows]
        np.save(os.path.join(directory, "log_prob_rows.npy"), rows.double().numpy())
    np.save(os.path.join(directory, "log_prob.npy"), lp.numpy())


def run_reference(args):
    """--impl reference: the reference's CPU path (oracle port; the Python reference itself cannot travel to the GPU box), on
    ALL host threads -- torchrun exports OMP_NUM_THREADS=1, undone here; ranks other than 0 exit without work."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    torch.set_num_threads(host_threads())
    flow = build_flow()
    rates, rows_total = [], 0
    for i in range(args.warmup + args.steps):
        r, rows, threads = cpu_oracle_rate(flow, budget_s=args.ref_budget, max_rows=args.ref_rows)
        if i >= args.warmup:
            rates.append(r)
            rows_total += rows
    value = sum(rates) / len(rates)
    sample = "{} rows per step in chunks of 2048 (of the {}-row workload)".format(rows_total // max(1, args.steps), args.rows)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * (rows_total / max(1, args.steps)) / value, "higher_is_better": True,
        "scaling": "weak" if args.weak else "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, world),
        "cpu_baseline": {"value": value, "unit": "samples/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def run_native(args):
    import torch.distributed as dist

    from nflows_b200 import _native
    from nflows_b200 import kernels as K

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    peaks = load_peaks()

    flow = build_flow().to(dev)
    rows = args.rows if args.weak else args.rows // world          # rows this rank owns
    gen = torch.Generator(device=dev).manual_seed(1 + rank)
    x = torch.randn(rows, FEATURES, device=dev, generator=gen)
    gathered = torch.empty(world * rows, device=dev) if world > 1 else None

    def step(inp):
        lp = flow.log_prob(inp)
        if world > 1:
            dist.all_gather_into_tensor(gathered, lp)
            return gathered
        return lp

    def fence():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.no_grad():
        for _ in range(args.warmup):
            step(x)
        # ---- device-resident timing ----------------------------------------------------------------------------
        sampler = ClockSampler(local)
        fence()
        if rank == 0:
            sampler.start()
        launches0 = _native.launch_count()
        K.TIMELINE = [] if rank == 0 else None
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            out = step(x)
        e1.record()
        fence()
        timeline, K.TIMELINE = K.TIMELINE, None
        launches = _native.launch_count() - launches0
        clocks = sampler.stop() if rank == 0 else None
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        ms_total = float(ms.item())
        lp_local = out[rank * rows:(rank + 1) * rows].clone() if world > 1 else out.clone()
        last_out = out.cpu() if args.dump_outputs and rank == 0 else None

        # ---- end to end: pinned host inputs -> H2D -> log_prob -> D2H of the result, every step ------------------
        host_x = torch.empty(rows, FEATURES, pin_memory=True)
        host_x.copy_(x)
        host_out = torch.empty(out.numel(), pin_memory=True)
        e2e_steps = args.steps
        from nflows_b200 import sharding
        lp_dev = torch.empty(rows, device=dev)
        sharding.log_prob_streamed(flow, host_x, dev, chunk_rows=args.e2e_chunk, out=lp_dev)       # warm-up (pinned staging, streams)
        fence()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for _ in range(e2e_steps):
            sharding.log_prob_streamed(flow, host_x, dev, chunk_rows=args.e2e_chunk, out=lp_dev)   # H2D overlapped with the kernels
            if world > 1:
                dist.all_gather_into_tensor(gathered, lp_dev)
                host_out.copy_(gathered, non_blocking=True)
            else:
                host_out.copy_(lp_dev, non_blocking=True)
        f1.record()
        fence()
        ms2 = torch.tensor([f0.elapsed_time(f1)], device=dev)
        if world > 1:
            dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
        e2e_ms = float(ms2.item()) / e2e_steps

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    ms_per_step = ms_total / args.steps
    value = world * rows / (ms_per_step * 1e-3)
    config = workload_config(args, world)          # identical in the reference arm's line
    result = {
        "metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak" if args.weak else "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": config,
        "clocks": clocks, "gpu_launches": int(launches),
        "e2e": {"value": world * rows / (e2e_ms * 1e-3), "unit": "samples/s", "h2d_bytes_per_step": rows * FEATURES * 4,
                "d2h_bytes_per_step": int(out.numel()) * 4, "ms_per_step": e2e_ms, "steps": e2e_steps},
        "tflops_effective": FLOP_PER_SAMPLE * value / 1e12,
        "notes": {"peaks": peaks["source"],
                  "arithmetic": "fp32 in / fp32 out; dense layers multiply fp16 (hi,lo) split pairs with 3 tcgen05 kind::f16 MMAs "
                                "per product (22-bit operands) and accumulate in fp32"},
    }
    # ---- parity of the timed result: random rows of the batch just timed against the CPU oracle -----------------------------
    if not args.no_parity_check:
        from oracle import flow_oracle as O
        g = torch.Generator().manual_seed(11)
        idx = torch.randperm(rows, generator=g)[:args.parity_rows].sort().values
        xs = x[idx.to(dev)].cpu()
        sd = {k: v.detach().cpu().clone() for k, v in flow.state_dict().items()}
        with torch.no_grad():
            want = O.flow_log_prob(sd, O.nsf_spec(LAYERS, num_bins=BINS, tail_bound=3.0), xs)
        got = lp_local[idx.to(dev)].cpu()
        finite = bool(torch.isfinite(lp_local).all().item())
        rel = float(((got - want).abs() / torch.maximum(torch.maximum(got.abs(), want.abs()), torch.ones_like(want))).max())
        result["parity_check"] = {"rows": int(idx.numel()), "of_rows": rows, "rel_err": rel, "tolerance": 1e-5, "all_finite": finite,
                                  "against": "oracle/flow_oracle.py (CPU fp32 restatement of the reference, pinned to reference goldens)",
                                  "ok": bool(finite and rel <= 1e-5)}
    # ---- roofline of the dominant kernel, timed live with CUDA events -------------------------------------------------------
    if timeline:
        torch.cuda.synchronize()
        tags = {}
        for tag, rows_k, a, b in timeline:
            t = tags.setdefault(tag, [0.0, 0, 0])
            t[0] += a.elapsed_time(b)
            t[1] += 1
            t[2] += rows_k
        result["timeline_ms_per_step"] = {k: round(v[0] / args.steps, 3) for k, v in sorted(tags.items(), key=lambda kv: -kv[1][0])}
        top = max(tags.items(), key=lambda kv: kv[1][0])
        tag, (tms, count, rows_k) = top
        per_row = {"rq_coupling_step": FLOP_COND_PER_ROW, "rq_coupling_final": FLOP_FINAL_PER_ROW}.get(tag, FLOP_AFFINE_PER_ROW)
        exec_per_row = {"rq_coupling_step": MMA_EXEC_STEP_PER_ROW, "rq_coupling_final": 3.0 * FLOP_FINAL_PER_ROW * FUSED_PAD}.get(
            tag, 3.0 * 2 * 800 * 832)
        achieved = per_row * rows_k / (tms * 1e-3) / 1e12
        peak = peaks["bf16_tflops_sustained"]
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
        if os.path.exists(tpath):
            t = json.load(open(tpath))
            t = t.get(tag, t) if isinstance(t.get(tag, None), dict) else t
            if t.get("kernel") == tag and "dram_bytes_per_row" in t:
                traffic = t["dram_bytes_per_row"] * (rows_k // count)     # per launch, like `achieved`
        result["roofline"] = {"kernel": tag, "bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                              "frac": achieved / peak, "traffic": traffic, "launches": count,
                              "avg_launch_ms": tms / count, "share_of_step": tms / ms_total,
                              "peak_kind": "bf16 dense sustained, %s" % peaks["source"],
                              "mma_tflops_executed": exec_per_row * rows_k / (tms * 1e-3) / 1e12,
                              "algorithmic_flop_per_row": per_row,
                              "note": "achieved counts ALGORITHMIC flops (2 per weight per row); the kernel executes 3 "
                                      "fp16 MMAs per algorithmic multiply-add plus tile padding (mma_tflops_executed)"}
        result["roofline_step"] = {"bound": "tensor", "achieved": FLOP_PER_SAMPLE * value / world / 1e12, "peak": peak, "unit": "TFLOP/s",
                                   "frac": FLOP_PER_SAMPLE * value / world / 1e12 / peak, "what": "whole log_prob step, algorithmic flops, per GPU"}
    if not args.no_spline_roofline:
        result["roofline_spline"] = spline_hbm_roofline(dev, peaks)
    if world == 1 and not args.no_extras:
        result["extra"] = extra_workloads(dev, flow)
    # ---- CPU baseline (oracle port) on this box's host cores ---------------------------------------------------
    if world == 1 and not args.no_cpu_baseline:
        try:
            best, tried = torch_cuda_rate(flow, dev)
            result["torch_cuda_baseline"] = {"value": best[0], "unit": "samples/s", "kind": "port", "chunk_rows": best[1],
                                             "chunk_sweep_samples_per_s": tried,
                                             "sample": "%d rows in chunks of %d (best of the sweep), torch eager fp32 (allow_tf32 off) on "
                                                       "the same GPU" % (best[2], best[1])}
        except Exception as exc:     # a context figure only: never let it take the bench line down
            result["torch_cuda_baseline"] = {"unavailable": "%s: %s" % (type(exc).__name__, exc)}
        torch.set_num_threads(host_threads())
        rate, sample_rows, threads = cpu_oracle_rate(flow.cpu(), budget_s=args.ref_budget, max_rows=args.ref_rows)
        result["cpu_baseline"] = {"value": rate, "unit": "samples/s", "cores": threads, "kind": "port",
                                  "sample": "%d rows of the same workload in chunks of 2048" % sample_rows}
    print(json.dumps(result))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last_out)
    if world > 1:
        dist.destroy_process_group()
    if "parity_check" in result and not result["parity_check"]["ok"]:
        sys.exit("parity check failed: %r" % (result["parity_check"],))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--rows", type=int, default=1 << 20, help="rows of the batch (BASELINE: 2^20), sharded over the GPUs")
    ap.add_argument("--weak", action="store_true", help="weak scaling: every GPU owns --rows rows")
    ap.add_argument("--ref-budget", type=float, default=12.0, help="seconds of CPU work per reference step")
    ap.add_argument("--ref-rows", type=int, default=1 << 15)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity-check", action="store_true")
    ap.add_argument("--parity-rows", type=int, default=512)
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--block-rows", type=int, default=0, help="override config.{trunk,affine,coupling}_block_rows (experiments)")
    ap.add_argument("--no-spline-roofline", action="store_true")
    ap.add_argument("--e2e-chunk", type=int, default=1 << 17, help="rows per host->device chunk of the end-to-end leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the log-probs of the last timed step to DIR/log_prob.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs applies to --impl native")
    if args.block_rows:
        from nflows_b200 import config
        config.trunk_block_rows = config.affine_block_rows = config.coupling_block_rows = args.block_rows
    if args.impl == "reference":
        run_reference(args)
    else:
        run_native(args)


if __name__ == "__main__":
    main()
