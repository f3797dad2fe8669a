// prof.cuh - measurement hooks: a launch counter (always on) and optional CUDA-event timing per
// kernel class, read by bench.py to report gpu_launches and the live roofline of the dominant kernel.
#pragma once
#include <cuda_runtime.h>
#include <atomic>
#include <mutex>
#include <vector>
#include <cstdint>

enum KClass {
    KC_SGEMM = 0, KC_GATES_FWD, KC_GATES_BWD, KC_HEAD, KC_LOSS, KC_OPTIM, KC_GATHER, KC_MISC,
    KC_TC_GEMM, KC_TC_SCAN_FWD, KC_TC_SCAN_BWD, KC_PACK, KC_TC_GEMM_DX, KC_TC_GEMM_DWIH, KC_TC_GEMM_DWHH, KC_INFER, KC_COUNT
};
static const char* const kKClassNames[KC_COUNT] = {
    "sgemm_f32", "gru_gates_fwd", "gru_gates_bwd", "head", "loss", "clip_adam", "window_gather", "misc",
    "tc_gemm_proj", "tc_gru_scan_fwd", "tc_gru_scan_bwd", "pack_bf16", "tc_gemm_dx", "tc_gemm_dwih", "tc_gemm_dwhh", "infer_cluster_scan"};

struct ProfRec { int cls; double flops, bytes; cudaEvent_t a, b; };
struct Profiler {
    std::atomic<long long> launches{0};
    std::atomic<int> enabled{0};
    std::mutex mu;
    std::vector<ProfRec> recs;
};
inline Profiler& profiler() { static Profiler p; return p; }

struct ProfScope {
    bool timed; ProfRec r; cudaStream_t st;
    ProfScope(int cls, double flops, double bytes, cudaStream_t s, int n_launches = 1) : timed(false), st(s) {
        Profiler& p = profiler();
        p.launches.fetch_add(n_launches, std::memory_order_relaxed);
        if (p.enabled.load(std::memory_order_relaxed)) {
            r.cls = cls; r.flops = flops; r.bytes = bytes;
            if (cudaEventCreate(&r.a) == cudaSuccess && cudaEventCreate(&r.b) == cudaSuccess) {
                cudaEventRecord(r.a, st);
                timed = true;
            }
        }
    }
    ~ProfScope() {
        if (timed) {
            cudaEventRecord(r.b, st);
            Profiler& p = profiler();
            std::lock_guard<std::mutex> g(p.mu);
            p.recs.push_back(r);
        }
    }
};
