// infer_cluster.cuh - the live predictor's eval-mode forward for models the single-CTA kernel (infer_small.cuh) cannot
// hold: long windows and hidden sizes up to 512.  Exact fp32 (FFMA, expf, tanhf), same gate / bias order as
// infer_window_kernel and gru_gates_fwd_kernel.  Per layer the host enqueues
//   1. the input projection of all T steps at once (sgemm_launch of kernels_f32.cuh: gi = x W_ih^T + b_ih), then
//   2. infer_cluster_scan_kernel: one thread-block cluster per (direction, group of G windows) walks the T steps.  CTA c
//      owns hidden units [c*U, c*U + U) and keeps their W_hh rows (3 gates x U x Hp fp32) in shared memory for the whole
//      scan.  Every CTA holds the full h_{t-1} of its G windows (double-buffered by step parity); after the gate math it
//      sends its new U-unit slice to every CTA of the cluster with st.async, which completes bytes on the receiver's
//      mbarrier of that parity.  The receiver arms that barrier with the G*Hp*4 bytes a step brings in and waits on it
//      before the next step: one all-to-all exchange per step, no cluster-wide barrier inside the loop.
// and after the top layer infer_head_kernel (pooling head + Linear + sigmoid, as infer_window_kernel).
#pragma once
#include "common.cuh"
#include "tc_common.cuh"
#include "infer_small.cuh"

namespace icl {

constexpr int kThreads = 512;
constexpr int kWarps = kThreads / 32;
constexpr int kUnitsPerWarp = 2;
constexpr int kMaxUnits = kWarps * kUnitsPerWarp;       // units one CTA can own (U <= 32)
constexpr int kMaxCluster = 16;                         // non-portable above 8
constexpr int kMaxHidden = kMaxCluster * kMaxUnits;     // 512

// shared memory of one CTA: 2 mbarriers | W_hh slice [3][U][Hp] | h [2][G][Hp] | outgoing slice [2][G][U]
__host__ __device__ inline size_t scan_smem_bytes(int U, int Hp, int G) {
    return 16 + sizeof(float) * (3 * (size_t)U * Hp + 2 * (size_t)G * Hp + 2 * (size_t)G * U);
}

// gi [D][B*T][3H] (b_ih included), Y [B][T][D*H].  Grid (NC, groups, D), cluster (NC, 1, 1), kThreads threads.
// U is a multiple of 4 and Hp = NC*U >= H; units >= H and k >= H are zero padding.
template <int G>
__global__ void __launch_bounds__(kThreads, 1)
infer_cluster_scan_kernel(const float* __restrict__ gi, const float* __restrict__ w_hh0, const float* __restrict__ b_hh0,
                          int64_t dir_stride, float* __restrict__ Y, int B, int T, int H, int D, int U) {
    extern __shared__ __align__(16) unsigned char ism_raw[];
    uint64_t* full = reinterpret_cast<uint64_t*>(ism_raw);
    const int NC = gridDim.x, Hp = NC * U;
    float* wsm = reinterpret_cast<float*>(ism_raw + 16);
    float* hbuf = wsm + 3 * (size_t)U * Hp;
    float* stg = hbuf + 2 * (size_t)G * Hp;
    const int c = blockIdx.x, grp = blockIdx.y, d = blockIdx.z;   // the cluster spans gridDim.x: c is the CTA rank
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const float* w_hh = w_hh0 + (int64_t)d * dir_stride;
    const float* b_hh = b_hh0 + (int64_t)d * dir_stride;
    const int u0 = c * U;
    for (int i = tid; i < 3 * U * Hp; i += kThreads) {
        const int k = i % Hp, ul = (i / Hp) % U, q = i / (Hp * U), u = u0 + ul;
        wsm[i] = (u < H && k < H) ? w_hh[((int64_t)q * H + u) * H + k] : 0.f;
    }
    for (int i = tid; i < 2 * G * Hp; i += kThreads) hbuf[i] = 0.f;          // h_0 = 0
    if (tid == 0) {
        tc::mbar_init(&full[0], 1);
        tc::mbar_init(&full[1], 1);
        tc::fence_mbar_init();
    }
    float bh[kUnitsPerWarp][3];
#pragma unroll
    for (int j = 0; j < kUnitsPerWarp; ++j) {
        const int u = u0 + warp + kWarps * j;
#pragma unroll
        for (int q = 0; q < 3; ++q) bh[j][q] = u < H ? b_hh[q * H + u] : 0.f;
    }
    __syncthreads();
    tc::cluster_sync_all();                     // every barrier of the cluster is initialised before the first st.async

    const int b_own = grp * G + lane;           // lanes < G do the gate math of window b_own
    const bool gate_lane = lane < G && b_own < B;
    const int DH = D * H;
    const uint32_t step_bytes = (uint32_t)(G * Hp * sizeof(float));
    const int chunks = G * U / 4;               // 16-byte pieces of the outgoing slice, per receiver
    for (int s = 0; s < T; ++s) {
        const int t = d == 0 ? s : T - 1 - s;
        const int cur = s & 1, nxt = cur ^ 1;
        // this step's input projection: independent of the recurrence, loaded before the wait so it overlaps it
        float x[kUnitsPerWarp][3];
#pragma unroll
        for (int j = 0; j < kUnitsPerWarp; ++j) {
            const int u = u0 + warp + kWarps * j;
            const float* g = gi + (((int64_t)d * B + b_own) * T + t) * 3 * H;
#pragma unroll
            for (int q = 0; q < 3; ++q) x[j][q] = (gate_lane && u < H) ? g[q * H + u] : 0.f;
        }
        if (s > 0) tc::mbar_wait_cluster(&full[cur], ((s - 1) >> 1) & 1, nullptr, 0x1C0u);
        if (tid == 0) tc::mbar_arrive_expect_tx(&full[nxt], step_bytes);   // the previous phase of full[nxt] completed at s-1
        const float* hc = hbuf + (size_t)cur * G * Hp;
        float* so = stg + (size_t)cur * G * U;
        // the warp's units share every h load: acc[j][gate][g] over lane-strided float4 columns, then a butterfly sum
        const int nu = warp + kWarps < U ? 2 : (warp < U ? 1 : 0);
        float acc[kUnitsPerWarp][3][G];
#pragma unroll
        for (int j = 0; j < kUnitsPerWarp; ++j)
#pragma unroll
            for (int q = 0; q < 3; ++q)
#pragma unroll
                for (int g = 0; g < G; ++g) acc[j][q][g] = 0.f;
        if (nu > 0) {
            for (int k = lane * 4; k < Hp; k += 128) {
                float4 h4[G];
#pragma unroll
                for (int g = 0; g < G; ++g) h4[g] = *reinterpret_cast<const float4*>(hc + (size_t)g * Hp + k);
#pragma unroll
                for (int j = 0; j < kUnitsPerWarp; ++j) {
                    if (j >= nu) break;
#pragma unroll
                    for (int q = 0; q < 3; ++q) {
                        const float4 w4 = *reinterpret_cast<const float4*>(wsm + ((size_t)q * U + warp + kWarps * j) * Hp + k);
#pragma unroll
                        for (int g = 0; g < G; ++g) {
                            float a = acc[j][q][g];
                            a = fmaf(w4.x, h4[g].x, a); a = fmaf(w4.y, h4[g].y, a); a = fmaf(w4.z, h4[g].z, a); a = fmaf(w4.w, h4[g].w, a);
                            acc[j][q][g] = a;
                        }
                    }
                }
            }
        }
#pragma unroll
        for (int j = 0; j < kUnitsPerWarp; ++j) {
            if (j >= nu) break;
            const int ul = warp + kWarps * j;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1)
#pragma unroll
                for (int q = 0; q < 3; ++q)
#pragma unroll
                    for (int g = 0; g < G; ++g) acc[j][q][g] += __shfl_xor_sync(0xffffffffu, acc[j][q][g], o);
            if (lane < G) {
                float sr = 0.f, sz = 0.f, sn = 0.f;
#pragma unroll
                for (int g = 0; g < G; ++g)
                    if (g == lane) { sr = acc[j][0][g]; sz = acc[j][1][g]; sn = acc[j][2][g]; }
                const int u = u0 + ul;
                const float r = infer_sigmoid(x[j][0] + (bh[j][0] + sr));
                const float z = infer_sigmoid(x[j][1] + (bh[j][1] + sz));
                const float n = tanhf(x[j][2] + r * (bh[j][2] + sn));
                const float hp = hc[(size_t)lane * Hp + u];
                float h = (1.f - z) * n + z * hp;
                if (u >= H || !gate_lane) h = 0.f;           // padded units and windows stay zero
                so[lane * U + ul] = h;
                if (gate_lane && u < H) Y[((int64_t)b_own * T + t) * DH + d * H + u] = h;
            }
        }
        __syncthreads();                        // the slice is complete; every read of hc for this step is done
        // publish h_{s+1}[units of this CTA] into buffer nxt of every CTA of the cluster (itself included)
        const uint32_t h_dst = tc::smem_u32(hbuf + (size_t)nxt * G * Hp + u0);
        const uint32_t bar = tc::smem_u32(&full[nxt]);
        for (int i = tid; i < NC * chunks; i += kThreads) {
            const int peer = i / chunks, ch = i % chunks, g = ch / (U / 4), q4 = ch % (U / 4);
            const uint4 v = *reinterpret_cast<const uint4*>(so + g * U + q4 * 4);
            tc::st_async_v4(tc::mapa_u32(h_dst + (uint32_t)((g * Hp + q4 * 4) * sizeof(float)), (uint32_t)peer), v,
                            tc::mapa_u32(bar, (uint32_t)peer));
        }
    }
    // every byte sent to this CTA has landed before any CTA of the cluster exits
    tc::mbar_wait_cluster(&full[T & 1], ((T - 1) >> 1) & 1, nullptr, 0x1C1u);
    tc::cluster_sync_all();
}

// pooling head (biGRU_model.py:111-137) + Linear + sigmoid of one window per CTA; same order as infer_window_kernel.
// Y [B][T][D*H] of the top layer; 3H floats of shared memory.
__global__ void infer_head_kernel(const float* __restrict__ Y, const float* __restrict__ lin_w, int T, int H, int C, int D,
                                  float* __restrict__ logits, float* __restrict__ probs) {
    extern __shared__ float cat[];
    const int b = blockIdx.x, DH = D * H;
    const float* y = Y + (int64_t)b * T * DH;
    for (int j = threadIdx.x; j < H; j += blockDim.x) {
        float last = y[(int64_t)(T - 1) * DH + j];            // h_n of the forward direction
        if (D == 2) last += y[H + j];                           // h_n of the reverse direction (t = 0)
        float mx = -INFINITY, sum = 0.f;
        for (int t = 0; t < T; ++t) {
            float sv = y[(int64_t)t * DH + j];
            if (D == 2) sv += y[(int64_t)t * DH + H + j];
            mx = fmaxf(mx, sv);
            sum += sv;
        }
        cat[j] = last; cat[H + j] = mx; cat[2 * H + j] = sum / (float)T;
    }
    __syncthreads();
    const float* lin_b = lin_w + 3LL * H * C;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        float v = lin_b[c];
        for (int k = 0; k < 3 * H; ++k) v = fmaf(cat[k], lin_w[(int64_t)c * 3 * H + k], v);
        logits[(int64_t)b * C + c] = v;
        if (probs) probs[(int64_t)b * C + c] = infer_sigmoid(v);
    }
}

}  // namespace icl
