"""Per-message latency of the live predictor for one window, at four model shapes: the shipped checkpoint (H 8, T 5,
F 108, L 1), the notebook model (H 32, T 30, F 108, L 2), BASELINE configs[1] (H 256, T 128, F 64, L 2) and configs[4]
(H 512, T 1024, F 128, L 2), all bidirectional with 4 labels, plus two shapes between them (H 64 / 128 at T 30) that
locate the crossover of LivePredictor's kernel choice.  Every route gets the same raw window:

  infer_window   bigru_infer_window (one CTA per window), where it accepts the shape
  infer_cluster  bigru_infer_cluster (SGEMM + cluster-resident scan per layer + head); at H 256 also capped to 8-CTA
                 clusters (BIGRU_INFER_CLUSTER_CTAS=8) to compare the cluster widths
  fp32_forward   BiGRU(precision="fp32").eval() forward (step-by-step launches) + sigmoid
  tc_forward     the tensor-core forward at B 1: precision="bf16x3" (H <= 256), "bf16" at H 512
  predict_wall   host wall time of LivePredictor.predict() including the D2H copy of the probabilities

Device times are CUDA events over N back-to-back calls after warm-up (N = 200, 20 for routes slower than 5 ms a call).
The scan's per-step time comes from a separate profiled pass (bigru_prof_*).  Records the GPU name, its power limit and
cudaOccupancyMaxActiveClusters of the cluster launches, read in the same run.

    python tools/bench_live_predictor.py [--out FILE.json]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from financial_market_data_analysis_b200 import BiGRU, _lib                # noqa: E402
from financial_market_data_analysis_b200.predict import SINGLE_CTA_MAX_HIDDEN, LivePredictor   # noqa: E402

SHAPES = [  # name, H, T, F, L
    ("shipped_checkpoint", 8, 5, 108, 1),
    ("notebook_model", 32, 30, 108, 2),
    ("h64_t30", 64, 30, 108, 2),
    ("h128_t30", 128, 30, 108, 2),
    ("configs1", 256, 128, 64, 2),
    ("configs4", 512, 1024, 128, 2),
]


def timed_us(fn, n=200):
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    if e0.elapsed_time(e1) > 5.0:
        n = 20
    for _ in range(10):
        fn()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return round(e0.elapsed_time(e1) / n * 1e3, 2), n


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=index,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else None
    except (OSError, subprocess.SubprocessError):
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    lib = _lib.load()
    dev = torch.device("cuda")
    stream = lambda: torch.cuda.current_stream().cuda_stream             # noqa: E731
    res = {"gpu": torch.cuda.get_device_name(), "power_limit_W,max_sm_clock": power_limit(),
           "single_cta_max_hidden": SINGLE_CTA_MAX_HIDDEN, "shapes": []}
    for name, H, T, F, L in SHAPES:
        Cn = 4
        torch.manual_seed(0)
        m = BiGRU(H, F, Cn, L, 50, 0.0, False, True, precision="fp32").to(dev).eval()
        state = {k: v.detach().cpu() for k, v in m.state_dict().items()}
        rng = np.random.default_rng(1)
        mn = rng.uniform(-5, 5, F).astype(np.float32)
        mx = (mn + rng.uniform(1, 10, F)).astype(np.float32)
        raw = (mn + rng.uniform(0, 1, (T, F)) * (mx - mn)).astype(np.float32)
        lp = LivePredictor(state, (mn, mx), window=T)
        x = torch.from_numpy(raw).to(dev)[None].contiguous()
        pp = m.flat_parameters()
        logits = torch.empty(1, Cn, device=dev)
        probs = torch.empty(1, Cn, device=dev)
        row = {"name": name, "H": H, "T": T, "F": F, "L": L, "bidirectional": True,
               "predictor_route": "infer_window" if H <= SINGLE_CTA_MAX_HIDDEN else "infer_cluster"}

        def win():
            return lib.bigru_infer_window(_lib.ptr(pp), _lib.ptr(x), _lib.ptr(lp.x_min), _lib.ptr(lp.x_max), 1, T, F, H, L, Cn, 1,
                                          _lib.ptr(logits), _lib.ptr(probs), stream())
        if win() == 0:
            row["infer_window_us"], row["infer_window_calls"] = timed_us(win)
        else:
            row["infer_window_us"] = "refused: " + lib.bigru_last_error().decode()

        nbytes = C.c_size_t()
        _lib.check(lib.bigru_infer_cluster_workspace_bytes(1, T, F, H, L, 1, C.byref(nbytes)), "workspace")
        work = torch.empty(nbytes.value // 4, dtype=torch.float32, device=dev)

        def clu():
            return lib.bigru_infer_cluster(_lib.ptr(pp), _lib.ptr(x), _lib.ptr(lp.x_min), _lib.ptr(lp.x_max), 1, T, F, H, L, Cn, 1,
                                           _lib.ptr(work), _lib.ptr(logits), _lib.ptr(probs), stream())
        caps = ["16", "8"] if H == 256 else ["16"]
        for cap in caps:
            os.environ["BIGRU_INFER_CLUSTER_CTAS"] = cap
            key = "infer_cluster" if cap == "16" else "infer_cluster_8cta"
            geo = [C.c_int() for _ in range(4)]
            rc = lib.bigru_infer_cluster_geometry(1, H, 1, *[C.byref(g) for g in geo])
            if rc != 0:
                row[key + "_us"] = "refused: " + lib.bigru_last_error().decode()
                continue
            row[key + "_geometry"] = dict(zip(("cluster_ctas", "units_per_cta", "windows_per_cluster", "max_active_clusters"),
                                              [g.value for g in geo]))
            _lib.check(clu(), "bigru_infer_cluster")
            row[key + "_us"], row[key + "_calls"] = timed_us(clu)
            lib.bigru_prof_enable(1)
            for _ in range(3):
                clu()
            torch.cuda.synchronize()
            ms, cnt, fl, by = C.c_double(), C.c_longlong(), C.c_double(), C.c_double()
            for k in range(lib.bigru_prof_classes()):
                if lib.bigru_prof_class_name(k) == b"infer_cluster_scan":
                    lib.bigru_prof_report(k, C.byref(ms), C.byref(cnt), C.byref(fl), C.byref(by))
            lib.bigru_prof_enable(0)
            row[key + "_scan_us_per_step"] = round(ms.value / max(cnt.value, 1) * 1e3 / T, 3)
        os.environ.pop("BIGRU_INFER_CLUSTER_CTAS", None)

        xn = ((x - lp.x_min) / (lp.x_max - lp.x_min)).contiguous()
        with torch.no_grad():
            row["fp32_forward_us"], row["fp32_forward_calls"] = timed_us(lambda: torch.sigmoid(m(xn)))
            tc = "bf16x3" if H <= 256 else "bf16"
            try:
                torch.manual_seed(0)
                mt = BiGRU(H, F, Cn, L, 50, 0.0, False, True, precision=tc).to(dev).eval()
                mt.load_state_dict(m.state_dict())
                us, n = timed_us(lambda: torch.sigmoid(mt(xn)))
                row["tc_forward"] = {"precision": tc, "us": us, "calls": n}
            except (ValueError, RuntimeError) as e:
                row["tc_forward"] = {"precision": tc, "error": str(e)[:200]}

        for _ in range(20):
            lp.predict(raw)
        n = 200 if H <= 256 else 50
        t0 = time.perf_counter()
        for _ in range(n):
            lp.predict(raw)
        row["predict_wall_us"], row["predict_calls"] = round((time.perf_counter() - t0) / n * 1e6, 2), n
        # the routes agree (fp32 parity class)
        ref = torch.sigmoid(m(xn)).detach()
        got = lp.forward_windows(raw)[1]
        row["max_abs_prob_diff_vs_fp32_forward"] = float((got - ref).abs().max())
        print(json.dumps(row), flush=True)
        res["shapes"].append(row)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
