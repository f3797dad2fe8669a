#!/usr/bin/env python
"""bench.py - sequences/sec of one biGRU train step on N B200s (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--precision bf16|fp32] [--dump-outputs DIR]
  N>1: python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N

--dump-outputs DIR writes what the last timed step of the headline returned, DIR/loss.npy and DIR/logits.npy (float32), so that
two builds run with the same arguments (same seeded inputs and initial parameters) can be compared output for output.  Compare
with a tolerance: the split-K reductions do not sum in a fixed order and Adam turns last-bit gradient differences into
lr-sized steps, so two runs of one build differ (NVIDIA B200, 1000 W limit, --steps 20 --warmup 5, two pairs of runs: loss
by up to 1.3e-4 relative, logits by up to 8e-3 of their largest magnitude).

A "step" is the body of the reference training loop (biGRU_model.py:198-210): zero_grad -> forward ->
CrossEntropy loss -> backward -> [gradient all-reduce] -> clip_grad_norm_(50) -> Adam, on the workload
BASELINE.json quotes the metric on: per-GPU batch 512, seq_len 128, 64 features, hidden 256, 2 layers,
bidirectional, 3 classes; weak scaling (per-GPU batch fixed, global batch = 512*N).
The headline (`value`, `e2e`, `roofline`) is measured on the precision that meets north_star's tolerance (logits <= 1e-4
rel of the reference's torch.nn.GRU path): "bf16x3", the fp32-class tensor-core path = BASELINE.json configs[1].  The
pure-bf16 tensor-core path (configs[2], logits ~3e-3) is measured in the same run and reported under `variants`.
Rank 0 prints ONE JSON line.  `--impl reference` times the reference's CPU implementation of the same
step (the oracle port: torch.nn.GRU on the host cores, as biGRU_model.py:54-56/:102 call it).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark writes nothing into the tree it runs from (which may be read-only)

METRIC = "sequences/sec (train step) biGRU h=256 seq=128 feat=64"
WORK = dict(per_gpu_batch=512, seq_len=128, n_features=64, hidden=256, layers=2, classes=3)
# --config c4: BASELINE.json configs[4] (long-sequence stress: persistent-kernel residency) - not the headline metric
WORK_C4 = dict(per_gpu_batch=256, seq_len=1024, n_features=128, hidden=512, layers=2, classes=3)
METRIC_C4 = "sequences/sec (train step) biGRU h=512 seq=1024 feat=128"


def flops_train_per_seq(T, F, H, L, C, D=2):
    """SURVEY.md 8(d): fwd = 12*T*H*sum_l(I_l+H) + 2*3H*C (bidirectional), train = 3x fwd."""
    fwd = 0
    for l in range(L):
        I = F if l == 0 else D * H
        fwd += 6 * D * T * H * (I + H)
    fwd += 2 * 3 * H * C
    return 3 * fwd


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                    if r[col].lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def synthetic(B, T, F, C, seed):
    import torch
    g = torch.Generator().manual_seed(seed)
    return torch.randn(B, T, F, generator=g), torch.randint(0, C, (B,), generator=g)


def host_cores():
    """Cores this process may actually use (affinity mask and cgroup quota, not the host's total)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    return max(1, n)


def time_cpu_reference(steps, warmup, budget_s=150.0):
    """The reference CPU path (oracle port) on the host cores, bounded sample of the same workload:
    a small calibration batch sizes the sample so that the whole call stays near budget_s."""
    import torch
    import torch.nn as nn
    from oracle.bigru_oracle import OracleBiGRU, train_step
    W = WORK
    cores = host_cores()
    torch.manual_seed(0)
    model = OracleBiGRU(W["hidden"], W["n_features"], W["classes"], W["layers"], 50, 0.0, False, True)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    loss_fn = nn.CrossEntropyLoss()
    model.train()
    xf, tf = synthetic(W["per_gpu_batch"], W["seq_len"], W["n_features"], W["classes"], 1234)
    cal = 32
    # "all the host threads it can use": more threads are not always faster for torch's CPU GRU (round 1: 96 threads were
    # slower than 16), so the calibration batch picks the fastest of a few thread counts and says which
    best = None
    for nt in sorted({min(cores, 8), min(cores, 16), min(cores, 32), cores}):
        torch.set_num_threads(nt)
        train_step(model, opt, loss_fn, xf[:cal].contiguous(), tf[:cal].contiguous())       # library warm-up
        t0 = time.perf_counter()
        train_step(model, opt, loss_fn, xf[:cal].contiguous(), tf[:cal].contiguous())
        dt0 = time.perf_counter() - t0
        if best is None or dt0 < best[0]:
            best = (dt0, nt)
    torch.set_num_threads(best[1])
    per_seq = best[0] / cal
    total = steps + max(warmup, 1)
    B = int(budget_s / (per_seq * total)) // 32 * 32
    B = max(32, min(W["per_gpu_batch"], B))
    x, t = xf[:B].contiguous(), tf[:B].contiguous()
    for _ in range(max(warmup, 1)):
        train_step(model, opt, loss_fn, x, t)
    t0 = time.perf_counter()
    for _ in range(steps):
        train_step(model, opt, loss_fn, x, t)
    dt = (time.perf_counter() - t0) / steps
    return {"value": B / dt, "unit": "sequences/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{steps} train steps of batch {B} x seq {W['seq_len']} x feat {W['n_features']} "
                      f"(hidden {W['hidden']}, {W['layers']} layers, bidirectional) through oracle/bigru_oracle.py "
                      f"(torch.nn.GRU CPU, {torch.get_num_threads()} threads - the fastest of the counts tried - of "
                      f"{cores} usable / {os.cpu_count()} host CPUs)",
            "ms_per_step": dt * 1e3, "batch": B}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = time_cpu_reference(args.steps, args.warmup)
    W = WORK
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": "sequences/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.gpus, "fp32", cpu=True, batch=r["batch"]),
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": r["value"], "unit": "sequences/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    _emit(line)


CONFIG_OF = {"bf16x3": "configs[1] (fused-gate tensor-core kernels at fp32 tolerance: split bf16x3 operands, fp32 accumulate)",
             "fp32": "configs[1] (fp32 FFMA parity path)", "bf16": "configs[2] (bf16 tcgen05 gate GEMM)"}
CONFIG_OF_C4 = {"bf16": "configs[4] (long sequence, hidden 512: 8-CTA-cluster persistent scans, bf16 tcgen05)",
                "fp32": "configs[4] (long sequence, hidden 512, fp32 FFMA path)"}


def workload_config(n_gpus, precision, cpu=False, batch=None):
    W = WORK
    b = batch or W["per_gpu_batch"]
    c4 = W["hidden"] == 512
    which = ("configs[4] shape" if c4 else "configs[0]/[1] shape") + " on the host CPU (reference arm)" if cpu else \
        (CONFIG_OF_C4 if c4 else CONFIG_OF).get(precision, "configs[4]" if c4 else "configs[1]")
    return {"workload": f"BASELINE.json {which}: biGRU train step, batch {W['per_gpu_batch']}/GPU x seq {W['seq_len']} x feat {W['n_features']}, "
                        f"hidden {W['hidden']}, {W['layers']} layers, bidirectional, 3-class cross-entropy, clip 50, Adam 1e-3",
            "global_batch": b * (1 if cpu else n_gpus), "per_gpu_batch": b, "seq_len": W["seq_len"],
            "n_features": W["n_features"], "hidden": W["hidden"], "layers": W["layers"], "bidirectional": True,
            "classes": W["classes"], "loss": "CrossEntropyLoss", "optimizer": "Adam(lr=1e-3)+clip_grad_norm_(50)",
            "parallelism": "cpu" if cpu else f"dp{n_gpus}", "precision": precision,
            "l2": "rotating input batches + >1 GB of activation traffic per step (>> 126 MB L2)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default=os.environ.get("BIGRU_B200_PRECISION", "auto"))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-variants", action="store_true", help="skip the secondary precision (bf16) measurement")
    ap.add_argument("--config", default="c1", choices=["c1", "c4"],
                    help="c1: BASELINE.json configs[1] (the headline metric); c4: configs[4] long sequence (B256 T1024 F128 H512)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the loss and logits of the headline's last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    global WORK, METRIC
    if args.config == "c4":
        WORK, METRIC = WORK_C4, METRIC_C4
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.nn as nn
    import torch.distributed as dist
    import financial_market_data_analysis_b200 as pkg
    from financial_market_data_analysis_b200.parallel import max_over_ranks
    from financial_market_data_analysis_b200.prefetch import DevicePrefetcher

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 path has no CPU fallback (use --impl reference for the CPU arm)")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("bench.py: --gpus N>1 must be launched with torch.distributed.run --nproc-per-node N")
        args.gpus = world
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = pkg._lib.load()
    C_ = pkg._lib.C
    W = WORK
    B, T, F, H, L, C = W["per_gpu_batch"], W["seq_len"], W["n_features"], W["hidden"], W["layers"], W["classes"]

    def plan_ok(code):
        h = C_.c_void_p()
        ok = lib.bigru_plan_create(B, T, F, H, L, C, 1, code, C_.byref(h)) == 0
        if ok:
            lib.bigru_plan_destroy(h)
        return ok

    precision = args.precision
    if precision == "auto":          # the path that meets the stated tolerance first
        precision = "bf16x3" if plan_ok(pkg._lib.PREC_BF16X3) else ("bf16" if plan_ok(pkg._lib.PREC_BF16) else "fp32")

    NBUF = 8 if args.config == "c1" else 2                    # c4: 134 MB per batch
    host = [synthetic(B, T, F, C, 1234 + rank + 97 * i) for i in range(NBUF)]
    host = [(x.pin_memory(), t.pin_memory()) for x, t in host]
    resident = [(x.to(dev), t.to(dev)) for x, t in host]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def make_model(prec):
        torch.manual_seed(0)                                    # same replica on every rank
        m = pkg.BiGRU(H, F, C, L, 50, 0.0, False, True, precision=prec).cuda()
        m.add_loss_fn(nn.CrossEntropyLoss())
        m.add_optimizer(torch.optim.Adam(m.parameters(), lr=1e-3))
        m.add_device(dev)
        m.train()
        if world > 1:
            m.enable_data_parallel()
        return m

    def timed(fn, steps, warmup):
        for i in range(warmup):
            fn(i)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0 = lib.bigru_launch_count()
        e0.record()
        for i in range(steps):
            fn(warmup + i)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        launches = lib.bigru_launch_count() - n0
        if world > 1:
            ms = max_over_ranks(ms, dev)
        return ms, launches

    def measure(prec, steps, warmup, with_e2e=True, with_roofline=True, clocks=False, keep_outputs=False):
        """value (device-resident inputs), e2e (pinned host inputs, H2D + loss D2H inside the timed region) and the live
        per-kernel-class roofline of one precision."""
        model = make_model(prec)
        out = {"precision": prec, "workload": (CONFIG_OF_C4 if args.config == "c4" else CONFIG_OF).get(prec)}
        last = [None]

        def step_resident(i):
            x, t = resident[i % NBUF]
            last[0] = model.train_step(x, t)

        sampler = ClockSampler(local)
        if clocks and rank == 0:
            sampler.start()
            time.sleep(0.3)
        ms, launches = timed(step_resident, steps, warmup)
        if clocks:
            out["clocks"] = sampler.stop() if rank == 0 else None
        if keep_outputs:
            out["_outputs"] = {k: v.float().cpu().numpy() for k, v in zip(("loss", "logits"), last[0])}
        ms_step = ms / steps
        out.update(value=B * world / (ms_step * 1e-3), ms_per_step=ms_step, gpu_launches=int(launches))
        if world > 1:
            # exposed communication: the same step with the gradient all-reduce switched off (replicas diverge harmlessly
            # for these few steps; a fresh model follows for every later arm)
            dpw = model._dp_world
            model._dp_world = 1
            ms0, _ = timed(step_resident, max(5, steps // 2), warmup)
            model._dp_world = dpw
            ms0 /= max(5, steps // 2)
            out["comm"] = {"ms_per_step_with_allreduce": ms_step, "ms_per_step_without": ms0,
                           "exposed_frac": max(0.0, 1.0 - ms0 / ms_step), "bytes_per_step": 4 * (model.flat_parameters().numel() + 1),
                           "collective": "one NCCL all_reduce(SUM) of the flat gradient + loss per step"}
            model = make_model(prec)

        if with_e2e:
            # Every step's inputs start in pinned host memory and are copied to the GPU inside the timed region
            # (DevicePrefetcher: side-stream copy ahead of use); every step's loss is read back to the host inside the
            # timed region (consumed LAG - 1 steps later, so a host hiccup does not drain the launch queue).
            LAG = 3
            loss_host = torch.zeros(LAG, dtype=torch.float32).pin_memory()
            last_loss = [0.0]

            def run_e2e(n):
                evs = [None] * LAG
                for i, (x, t) in enumerate(DevicePrefetcher((host[k % NBUF] for k in range(n)), dev, depth=LAG)):
                    k = i % LAG
                    if evs[k] is not None:
                        evs[k].synchronize()
                        last_loss[0] = float(loss_host[k])
                    loss, _ = model.train_step(x, t)
                    loss_host[k:k + 1].copy_(loss, non_blocking=True)
                    evs[k] = torch.cuda.Event()
                    evs[k].record()
                for j in range(LAG):
                    k = (n + j) % LAG
                    if evs[k] is not None:
                        evs[k].synchronize()
                        last_loss[0] = float(loss_host[k])

            run_e2e(warmup)
            reps = []
            for _ in range(3):                  # a host hiccup (other tenants on the box's cores) shows in a 60 ms region: best of 3
                barrier()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                run_e2e(steps)
                e1.record()
                barrier()
                ms_r = e0.elapsed_time(e1)
                if world > 1:
                    ms_r = max_over_ranks(ms_r, dev)
                reps.append(ms_r)
            ms_e = min(reps)
            # what the box's host -> device link gives right now (pinned, 128 MB): the full-batch arm needs
            # h2d_bytes_per_step * steps/s of it; a contended PCIe link shows here, not in the kernels
            probe_src = torch.empty(32 * 1024 * 1024, dtype=torch.float32).pin_memory()
            probe_dst = torch.empty_like(probe_src, device=dev)
            probe_dst.copy_(probe_src, non_blocking=True); torch.cuda.synchronize()
            p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            p0.record(); probe_dst.copy_(probe_src, non_blocking=True); p1.record(); torch.cuda.synchronize()
            h2d_gbps = probe_src.numel() * 4 / (p0.elapsed_time(p1) * 1e-3) / 1e9
            del probe_src, probe_dst
            out["e2e"] = {"value": B * world / (ms_e / steps * 1e-3), "unit": "sequences/s", "h2d_probe_gbps": h2d_gbps,
                          "h2d_bytes_per_step": host[0][0].numel() * 4 + host[0][1].numel() * 8, "d2h_bytes_per_step": 4,
                          "ms_per_step": ms_e / steps, "loss": last_loss[0], "ms_per_step_repetitions": [r / steps for r in reps],
                          "how": "BiGRU.train_step on DevicePrefetcher batches: pinned host -> device copy of every step's inputs on a "
                                 "side stream ahead of their use, every step's loss read back through a pinned ring and consumed by the "
                                 "host %d steps later (all reads complete inside the timed region); the region of `steps` steps is timed 3 times, the fastest is "
                                 "reported (all three in ms_per_step_repetitions)" % (LAG - 1)}

        if with_roofline:
            psteps = 3
            if rank == 0:
                lib.bigru_prof_enable(1)
            graphs_were = getattr(model, "use_cuda_graph", False)
            model.use_cuda_graph = False            # the per-kernel events are recorded by the launch wrappers: plain launches here
            for i in range(psteps):                 # every rank steps (the step contains the gradient all-reduce)
                step_resident(i)
            barrier()
            model.use_cuda_graph = graphs_were
            if rank == 0:
                rows = []
                for k in range(lib.bigru_prof_classes()):
                    a, n, fl, by = C_.c_double(), C_.c_longlong(), C_.c_double(), C_.c_double()
                    lib.bigru_prof_report(k, C_.byref(a), C_.byref(n), C_.byref(fl), C_.byref(by))
                    if n.value:
                        rows.append(dict(name=lib.bigru_prof_class_name(k).decode(), ms=a.value / psteps,
                                         launches=n.value // psteps, flops=fl.value / psteps, bytes=by.value / psteps))
                lib.bigru_prof_enable(0)
                rows.sort(key=lambda r: -r["ms"])
                peaks = {}
                try:
                    peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
                except Exception:
                    pass
                tf_peak = peaks.get("bf16_tflops_sustained") or 1400.0     # kernel timed inside a long step
                hbm_peak = peaks.get("hbm_gbs") or 6650.0
                src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"
                if rows:
                    top = rows[0]
                    if top["flops"] > 0:
                        ach = top["flops"] / (top["ms"] * 1e-3) / 1e12
                        rl = {"kernel": top["name"], "bound": "tensor", "achieved": ach, "peak": tf_peak, "unit": "TFLOP/s",
                              "frac": ach / tf_peak, "traffic": None, "peak_source": src + ", sustained bf16",
                              "ms_per_step_in_kernel": top["ms"], "launches_per_step": top["launches"]}
                    else:
                        ach = top["bytes"] / (top["ms"] * 1e-3) / 1e9
                        rl = {"kernel": top["name"], "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s",
                              "frac": ach / hbm_peak, "traffic": None, "peak_source": src,
                              "ms_per_step_in_kernel": top["ms"], "launches_per_step": top["launches"]}
                    if prec == "bf16x3":
                        rl["note"] = ("achieved = ALGORITHMIC FLOPs (SURVEY 8(d): 2*3H*H per row-step, 2*M*N*K per GEMM) over measured time, against "
                                      "the bf16 peak; the fp32-class products issue 4x (recurrence) / 3x (GEMMs) that many bf16 tensor FLOPs")
                    try:        # DRAM traffic of the dominant kernel from the committed ncu --set full capture (per launch)
                        tr = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
                        ent = tr.get(prec, {}).get(top["name"])
                        if ent:
                            rl["traffic"] = ent["dram_bytes_per_launch"]
                            rl["traffic_source"] = ent["source"]
                    except Exception:
                        pass
                    step_flops = flops_train_per_seq(T, F, H, L, C) * B
                    rl["step_model_tflops"] = step_flops / (ms_step * 1e-3) / 1e12
                    rl["step_frac_of_gemm_roofline"] = rl["step_model_tflops"] / tf_peak
                    rl["kernel_shares"] = [{"kernel": r["name"], "ms_per_step": round(r["ms"], 4), "launches": r["launches"]}
                                           for r in rows[:8]]
                    out["roofline"] = rl
        out["_model"] = model
        return out

    head = measure(precision, args.steps, args.warmup, clocks=True, keep_outputs=bool(args.dump_outputs))
    model = head.pop("_model")
    outputs = head.pop("_outputs", None)

    # ---- end to end THROUGH THE LOADER (SURVEY 8(f) N1): a host chunk -> device -> zero-copy windows ----------------
    e2e_windows = None
    try:
        from financial_market_data_analysis_b200.sql_pytorch_dataloader import MySQLBatchLoader
        g = torch.Generator().manual_seed(4321 + rank)
        n_rows = B + T - 1
        chunks = [(torch.rand(n_rows, F, generator=g).pin_memory(), torch.randint(0, C, (n_rows, 1), generator=g).float().pin_memory())
                  for _ in range(4)]
        xmin, xmax = torch.zeros(1, F), torch.ones(1, F) * 1.001
        dss = [MySQLBatchLoader.from_tensors(cx.to(dev), cy.to(dev), (xmin, xmax), window=T) for cx, cy in chunks]
        side = torch.cuda.Stream(device=dev)

        wl_host = torch.zeros(4, dtype=torch.float32).pin_memory()
        wl_ev = [None] * 4

        def step_windows(i):
            ds, (cx, cy) = dss[i % 4], chunks[i % 4]
            k = i % 4
            if wl_ev[k] is not None:
                wl_ev[k].synchronize()                         # the loss of 4 steps ago has reached the host
            with torch.cuda.stream(side):                      # this step's chunk: 164 KB host -> device
                ds.x_raw.copy_(cx, non_blocking=True)
                ds.y.copy_(cy, non_blocking=True)
            torch.cuda.current_stream(dev).wait_stream(side)
            loss, _ = model.train_step_windows(ds, 0, B)
            wl_host[k:k + 1].copy_(loss, non_blocking=True)    # every step's loss is read back (pinned ring, consumed 4 steps later)
            wl_ev[k] = torch.cuda.Event()
            wl_ev[k].record()
            side.wait_stream(torch.cuda.current_stream(dev))
            return loss

        ms_w, _ = timed(step_windows, args.steps, args.warmup)
        e2e_windows = {"value": B * world / (ms_w / args.steps * 1e-3), "unit": "sequences/s", "ms_per_step": ms_w / args.steps,
                       "h2d_bytes_per_step": n_rows * (F + 1) * 4, "d2h_bytes_per_step": 4,
                       "how": "host chunk (B+T-1 rows x F + targets, pinned) -> device copy inside the timed region -> BiGRU.train_step_windows: the "
                              "windowed collation, min-max normalisation and the cast are fused into the first kernel (no x[B,T,F] anywhere); "
                              "every step's loss is read back to the host through a pinned ring"}
    except Exception as e:                                      # the extra arm must never break the bench line
        e2e_windows = {"error": str(e)[:200]}

    # ---- the other tensor-core precision, same run (bf16 = configs[2]; fp32-class = configs[1]) -------------------
    variants = {}
    del model
    if not args.no_variants:
        other = "bf16" if precision != "bf16" else "bf16x3"
        code = {"bf16": pkg._lib.PREC_BF16, "bf16x3": pkg._lib.PREC_BF16X3}[other]
        if plan_ok(code):
            v = measure(other, max(5, args.steps // 2), args.warmup, with_e2e=True, with_roofline=True)
            v.pop("_model")
            variants[other] = v

    # ---- in-run parity of both tensor-core paths against the oracle (checker only; small batch of the same shape) ----
    parity = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            from oracle.bigru_oracle import OracleBiGRU
            torch.manual_seed(0)
            ref = OracleBiGRU(H, F, C, L, 50, 0.0, False, True)
            ref.eval()
            xs = host[0][0][:(64 if args.config == "c1" else 16)].contiguous()
            with torch.no_grad():
                want = ref(xs)
            parity = {"what": "max |logit - oracle logit| / max |oracle logit| on %d sequences of the benchmark shape (eval mode); "
                              "the full-batch figures with gradients are in profiles/r02_parity_c%s.json (tests/test_gpu_parity.py)"
                              % (xs.shape[0], "1" if args.config == "c1" else "4"),
                      "tolerance": 1e-4 if args.config == "c1" else 3e-2}
            for prec in [precision] + list(variants):
                m2 = pkg.BiGRU(H, F, C, L, 50, 0.0, False, True, precision=prec)
                m2.load_state_dict(ref.state_dict())
                m2 = m2.cuda().eval()
                with torch.no_grad():
                    got = m2(xs.to(dev)).cpu()
                parity[prec] = float((got - want).abs().max() / want.abs().max())
        except Exception as e:
            parity = {"error": str(e)[:200]}

    # ---- context only: the reference wrapper on torch's cuDNN GRU on this GPU (BASELINE config 1 comparator) ----
    cudnn = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            from oracle.bigru_oracle import OracleBiGRU, train_step as oracle_step
            torch.manual_seed(0)
            ref = OracleBiGRU(H, F, C, L, 50, 0.0, False, True).cuda()
            ropt = torch.optim.Adam(ref.parameters(), lr=1e-3)
            rloss = nn.CrossEntropyLoss()
            xr, tr_ = resident[0]
            for _ in range(3):
                oracle_step(ref, ropt, rloss, xr, tr_)
            torch.cuda.synchronize()
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record()
            for i in range(5):
                oracle_step(ref, ropt, rloss, *resident[i % NBUF])
            c1.record()
            torch.cuda.synchronize()
            cms = c0.elapsed_time(c1) / 5
            cudnn = {"value": B / (cms * 1e-3), "unit": "sequences/s", "ms_per_step": cms,
                     "what": "reference wrapper restated on torch.nn.GRU CUDA (cuDNN, fp32/TF32 defaults), same step, same shapes; "
                             "comparator only, not part of the product"}
            del ref, ropt
        except Exception as e:                              # the comparator must never break the bench line
            cudnn = {"error": str(e)[:200]}

    # ---- reference CPU path on this box's host cores (rank 0, N=1) -----------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        r = time_cpu_reference(steps=3, warmup=1, budget_s=20.0)
        cpu = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}

    if rank == 0:
        dt = {"bf16": "bf16", "bf16x3": "bf16x3 (fp32-class: split bf16 operand pairs on tensor cores, fp32 accumulate / state / gradients)",
              "fp32": "f32"}[precision]
        line = {"metric": METRIC, "value": head["value"], "unit": "sequences/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": dt, "data": "synthetic",
                "config": workload_config(world, precision), "clocks": head.get("clocks"), "e2e": head.get("e2e"),
                "gpu_launches": head["gpu_launches"], "roofline": head.get("roofline"), "cpu_baseline": cpu,
                "e2e_windows": e2e_windows, "variants": variants, "parity": parity, "cudnn_comparator": cudnn, "comm": head.get("comm")}
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
        _emit(line)
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(directory, arrays):
    """One DIR/<name>.npy per array."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def _emit(obj):
    """The ONE JSON line goes to the process's real stdout; everything libraries print meanwhile (NCCL's version banner
    lands on fd 1) was redirected to stderr by _guard_stdout."""
    os.write(_REAL_STDOUT, (json.dumps(obj) + "\n").encode())


def _guard_stdout():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


_REAL_STDOUT = 1

if __name__ == "__main__":
    _guard_stdout()
    main()
