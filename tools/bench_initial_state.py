"""Cost of an initial hidden state on the bf16 tensor-core path: BiGRU.train_step(x, y) against train_step(x, y, hidden) at
BASELINE.json configs[1] (B512 T128 F64 H256 L2) and configs[4] (B256 T1024 F128 H512 L2).

Both sides run as plain launches (use_cuda_graph = False: a step with `hidden` is never graph-captured, so a captured step
without it would not be a like-for-like comparison).  Every shape and variant is warmed up first; then timed windows of
`--steps` steps, bracketed by CUDA events, alternate between the two variants `--reps` times, so that drift on a shared
machine hits both alike.  The card's name and power limit are read in the same run.
GPU box:  python tools/bench_initial_state.py [--out profiles/r03_bf16_h0.json]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import financial_market_data_analysis_b200 as pkg  # noqa: E402

SHAPES = {"configs[1]": dict(B=512, T=128, F=64, H=256, L=2, C=3, steps=40),
          "configs[4]": dict(B=256, T=1024, F=128, H=512, L=2, C=3, steps=8)}


def card():
    q = "name,power.limit,clocks.max.sm,driver_version"
    try:
        row = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        row = f"nvidia-smi unavailable ({e})"
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": dict(zip(q.split(","), [v.strip() for v in row.split(",")]))}


def window_ms(m, x, y, h0, n):
    st = torch.cuda.current_stream()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(st)
    for _ in range(n):
        m.train_step(x, y, h0)
    b.record(st)
    b.synchronize()
    return a.elapsed_time(b) / n


def kernel_classes_ms(m, x, y, h0, n=3):
    """Device time per step of each kernel class (the library's per-launch CUDA events) over n steps - a separate pass: the
    events sit between the launches, so these are not the timed windows' numbers."""
    import ctypes as C_
    lib = pkg._lib.load()
    lib.bigru_prof_enable(1)
    for _ in range(n):
        m.train_step(x, y, h0)
    torch.cuda.synchronize()
    rows = {}
    for k in range(lib.bigru_prof_classes()):
        a, cnt, fl, by = C_.c_double(), C_.c_longlong(), C_.c_double(), C_.c_double()
        lib.bigru_prof_report(k, C_.byref(a), C_.byref(cnt), C_.byref(fl), C_.byref(by))
        if cnt.value:
            rows[lib.bigru_prof_class_name(k).decode()] = dict(ms=round(a.value / n, 4), launches=cnt.value // n)
    lib.bigru_prof_enable(0)
    return rows


def stats(v):
    return dict(median_ms=statistics.median(v), min_ms=min(v), max_ms=max(v), windows_ms=v)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5, help="timed windows per variant (alternating)")
    ap.add_argument("--warmup", type=int, default=3, help="untimed steps per variant and shape")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_bf16_h0.json"))
    args = ap.parse_args()
    torch.cuda.set_device(0)
    result = {"what": "BiGRU.train_step at precision='bf16', plain launches, without and with `hidden` ([L*D, B, H], randn * 0.5); "
                      "CE loss, Adam; ms per step from CUDA events over windows of `steps` steps, the two variants alternating",
              "card": card(), "shapes": {}}
    for name, s in SHAPES.items():
        B, T, F, H, L, C, n = s["B"], s["T"], s["F"], s["H"], s["L"], s["C"], s["steps"]
        torch.manual_seed(0)
        m = pkg.BiGRU(H, F, C, L, 50, 0.0, False, True, precision="bf16").cuda().train()
        m.use_cuda_graph = False
        m.add_loss_fn(nn.CrossEntropyLoss())
        m.add_optimizer(torch.optim.Adam(m.parameters(), lr=1e-4))
        g = torch.Generator().manual_seed(1)
        x = torch.randn(B, T, F, generator=g).cuda()
        y = torch.randint(0, C, (B,), generator=g).cuda()
        h0 = (torch.randn(L * 2, B, H, generator=g) * 0.5).cuda()
        variants = {"no_hidden": None, "hidden": h0}
        for v in variants.values():
            for _ in range(args.warmup):
                m.train_step(x, y, v)
        torch.cuda.synchronize()
        times = {k: [] for k in variants}
        for _ in range(args.reps):
            for k, v in variants.items():
                times[k].append(window_ms(m, x, y, v, n))
        row = dict(shape=dict(B=B, T=T, F=F, H=H, L=L, C=C), steps_per_window=n, **{k: stats(v) for k, v in times.items()})
        a, b = row["no_hidden"], row["hidden"]
        row["hidden_minus_no_hidden_ms"] = b["median_ms"] - a["median_ms"]
        row["hidden_over_no_hidden"] = b["median_ms"] / a["median_ms"]
        row["no_hidden_spread_ms"] = a["max_ms"] - a["min_ms"]
        row["kernel_classes_ms_per_step"] = {k: kernel_classes_ms(m, x, y, v) for k, v in variants.items()}
        result["shapes"][name] = row
        print(f"{name}: no hidden {a['median_ms']:.3f} ms [{a['min_ms']:.3f}, {a['max_ms']:.3f}]  hidden {b['median_ms']:.3f} ms "
              f"[{b['min_ms']:.3f}, {b['max_ms']:.3f}]  ratio {row['hidden_over_no_hidden']:.4f}", flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result["card"]))


if __name__ == "__main__":
    main()
