// path_bf16.cuh - BIGRU_PREC_BF16: the tensor-core path.
//   input projections, dX and weight gradients : tc_gemm.cuh  (tcgen05 + TMA, bf16 operands, fp32 accumulate)
//   recurrences forward / backward              : tc_scan.cuh  (persistent cluster kernels, W_hh resident in tensor memory)
//   head, loss glue, optimiser                  : the fp32 kernels of kernels_f32.cuh
// All activations inside this path are TIME-MAJOR (row r = t*B + b) so that one step of one batch tile is a
// contiguous block of rows.  Supported: H in {128, 256} with B % 16 == 0 and H = 512 with B % 32 == 0, any F (K extent padded
// to 8), with or without an initial hidden state; anything else fails with BIGRU_ERR_UNSUPPORTED (the fp32 path covers the
// general case).  An initial state enters as in path_x3.cuh: W_hh h0 is formed once per layer in fp32 (FFMA GEMM) and the scans
// read it at step 0, which has no recurrent MMA; the backward scans run one more product for d(h0).
#pragma once
#include "common.cuh"
#include "kernels_f32.cuh"
#include "tc_gemm.cuh"
#include "tc_scan.cuh"
#include "tc_scan_w.cuh"
#include <algorithm>

typedef __nv_bfloat16 bf16_t;

// hidden size 512 runs on the 8-CTA-cluster kernels of tc_scan_w.cuh (64-unit slices, 32-row batch tiles)
static inline bool bf16_wide(const bigru_plan& p) { return p.H == 512; }
static int bf16_plan_check(const bigru_plan& p) {
    const bool ok = ((p.H == 128 || p.H == 256) && p.B % 16 == 0) || (p.H == 512 && p.B % 32 == 0);
    if (!ok) {
        bigru_set_error("BIGRU_PREC_BF16 supports hidden_size 128 or 256 with batch %% 16 == 0 and hidden_size 512 with batch %% 32 == 0 "
                        "(got H=%d B=%d; the Python mirror pads other batch sizes with zero rows); use BIGRU_PREC_FP32 for other shapes", p.H, p.B);
        return BIGRU_ERR_UNSUPPORTED;
    }
    return BIGRU_OK;
}

struct Bf16Layout {            // byte offsets, 1024-aligned
    size_t Yrow[16], YB[16], G[16], Xrow[16];                    // stash: activations
    size_t Wih[16], WihT[16], Wimg[16], WTimg[16], bfold[16], bhn[16];   // stash: packed weights
    size_t cat, arg, dbg, stash_total;
    size_t gi, dghn, dYa, dYb, dcat, dhinit, gh0, scratch_total;
};
static inline size_t al(size_t x) { return (x + 1023) & ~(size_t)1023; }
// Layer-0 operands (X rows and W_ih rows) are stored with their K extent (n_features) padded to a multiple of 8 with zeros: a
// TMA row pitch must be a multiple of 16 bytes.  The padding never leaves the packed images (gradients keep n_features columns).
static inline int pad8(int64_t v) { return (int)((v + 7) & ~(int64_t)7); }
static Bf16Layout bf16_layout(const bigru_plan& p) {
    Bf16Layout L{};
    const size_t R = (size_t)p.B * p.T, DH = (size_t)p.D * p.H, H = p.H, D = p.D;
    size_t o = 0;
    for (int l = 0; l < p.L; ++l) {
        const size_t I = p.in_size(l), Ip = (size_t)pad8((int64_t)I);
        L.Yrow[l] = o; o = al(o + R * DH * 2);
        L.YB[l] = o; o = al(o + R * DH * 2);
        L.G[l] = o; o = al(o + R * D * 4 * H * 2);
        L.Xrow[l] = o; o = al(o + R * Ip * 2);
        L.Wih[l] = o; o = al(o + D * 3 * H * Ip * 2);
        L.WihT[l] = o; o = al(o + D * 3 * H * I * 2);
        L.Wimg[l] = o; o = al(o + D * (bf16_wide(p) ? 4 : 3) * H * H * 2);     // wide: [CS][128][H + 384] TMEM image + [CS][2][128][64] tail
        L.WTimg[l] = o; o = al(o + D * 3 * H * H * 2);
        L.bfold[l] = o; o = al(o + D * 3 * H * 4);
        L.bhn[l] = o; o = al(o + D * H * 4);
    }
    L.cat = o; o = al(o + (size_t)p.B * 3 * H * 4);
    L.arg = o; o = al(o + (size_t)p.B * H * 4);
    L.dbg = o; o = al(o + 256);
    L.stash_total = o;
    o = 0;
    const size_t wide = DH > (size_t)p.F ? DH : (size_t)p.F;
    L.gi = o; o = al(o + R * D * 3 * H * 2);
    L.dghn = o; o = al(o + R * D * H * 2);
    L.dYa = o; o = al(o + R * wide * 4);
    L.dYb = o; o = al(o + R * wide * 4);
    L.dcat = o; o = al(o + (size_t)p.B * 3 * H * 4);
    L.dhinit = o; o = al(o + D * (size_t)p.B * H * 4);
    L.gh0 = o; o = al(o + (size_t)p.B * D * 3 * H * 4);          // W_hh h0 of the layer being scanned (initial state given)
    L.scratch_total = o;
    return L;
}
static void bf16_workspace(const bigru_plan& p, size_t* a, size_t* b) {
    const Bf16Layout L = bf16_layout(p);
    *a = L.stash_total; *b = L.scratch_total;
}

// ---------------------------------------------------------------------------------------------------
// small kernels of this path
// ---------------------------------------------------------------------------------------------------
// x fp32 [B][T][F] -> Xrow bf16 [(t*B+b)][F] (time-major rows), optional input dropout.  With `src` set the batch is
// read straight from the chunk table: x[b,t,f] = (src[start+b+t, f] - xmin[f]) / (xmax[f] - xmin[f])  (zero-copy windows).
struct WindowSrc { const float* src; const float* xmin; const float* xmax; int64_t start; };
__global__ void cast_x_kernel(const float* __restrict__ x, WindowSrc w, bf16_t* __restrict__ Xrow, bf16_t* __restrict__ Xlo, int B, int T, int F,
                              float pdrop, int spatial, uint64_t seed) {
    const float scale = pdrop > 0.f ? 1.f / (1.f - pdrop) : 1.f;
    const int F4 = F >> 2;                          // F % 8 == 0 on the tensor-core path
    const int64_t total = (int64_t)B * T * F4;
    const int64_t nthr = (int64_t)gridDim.x * blockDim.x;
    constexpr int U = 4;                            // loads in flight per thread (the kernel is pure latency otherwise)
    for (int64_t i0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i0 < total; i0 += U * nthr) {
        float4 v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int64_t i = i0 + u * nthr;
            if (i >= total) break;
            const int f = (int)(i % F4) * 4;
            const int64_t r = i / F4;                // output row t*B + b
            const int64_t b = r % B, t = r / B;
            v[u] = w.src ? *reinterpret_cast<const float4*>(w.src + (w.start + b + t) * F + f)
                         : *reinterpret_cast<const float4*>(x + (b * T + t) * F + f);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int64_t i = i0 + u * nthr;
            if (i >= total) break;
            const int f = (int)(i % F4) * 4;
            const int64_t r = i / F4;
            const int64_t b = r % B, t = r / B;
            float4 q = v[u];
            if (w.src && w.xmin) {
                const float4 mn = *reinterpret_cast<const float4*>(w.xmin + f), mx = *reinterpret_cast<const float4*>(w.xmax + f);
                q.x = (q.x - mn.x) / (mx.x - mn.x); q.y = (q.y - mn.y) / (mx.y - mn.y);
                q.z = (q.z - mn.z) / (mx.z - mn.z); q.w = (q.w - mn.w) / (mx.w - mn.w);
            }
            if (pdrop > 0.f) {
                float* e = &q.x;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const uint64_t key = spatial ? (uint64_t)b * F + f + k : ((uint64_t)b * T + t) * F + f + k;
                    e[k] = bigru_uniform(seed, 0u, key) < pdrop ? 0.f : e[k] * scale;
                }
            }
            __nv_bfloat162 lo = __floats2bfloat162_rn(q.x, q.y), hi = __floats2bfloat162_rn(q.z, q.w);
            *reinterpret_cast<uint2*>(Xrow + r * F + f) = make_uint2(*reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi));
            if (Xlo) {          // x3 path: the residuals x - bf16(x), again as bf16
                const float2 a = __bfloat1622float2(lo), b2 = __bfloat1622float2(hi);
                __nv_bfloat162 rl = __floats2bfloat162_rn(q.x - a.x, q.y - a.y), rh = __floats2bfloat162_rn(q.z - b2.x, q.w - b2.y);
                *reinterpret_cast<uint2*>(Xlo + r * F + f) = make_uint2(*reinterpret_cast<uint32_t*>(&rl), *reinterpret_cast<uint32_t*>(&rh));
            }
        }
    }
}

// the same for n_features % 8 != 0: element-wise, rows written with the padded pitch Fp = pad8(F) (zero columns behind F)
__global__ void cast_x_pad_kernel(const float* __restrict__ x, WindowSrc w, bf16_t* __restrict__ Xrow, bf16_t* __restrict__ Xlo, int B, int T, int F,
                                  int Fp, float pdrop, int spatial, uint64_t seed) {
    const float scale = pdrop > 0.f ? 1.f / (1.f - pdrop) : 1.f;
    const int64_t total = (int64_t)B * T * Fp;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int f = (int)(i % Fp);
        const int64_t r = i / Fp;
        const int64_t b = r % B, t = r / B;
        float v = 0.f;
        if (f < F) {
            if (w.src) {
                v = w.src[(w.start + b + t) * F + f];
                if (w.xmin) v = (v - w.xmin[f]) / (w.xmax[f] - w.xmin[f]);
            } else {
                v = x[(b * T + t) * F + f];
            }
            if (pdrop > 0.f) {
                const uint64_t key = spatial ? (uint64_t)b * F + f : ((uint64_t)b * T + t) * F + f;
                v = bigru_uniform(seed, 0u, key) < pdrop ? 0.f : v * scale;
            }
        }
        const bf16_t h = __float2bfloat16(v);
        Xrow[i] = h;
        if (Xlo) Xlo[i] = __float2bfloat16(v - __bfloat162float(h));
    }
}

// zero-copy windows (SURVEY.md 8(f) N1): the chunk rows [start, start + rows) are normalised and cast ONCE ((B+T-1) x F
// values instead of B*T*F); the kernels that consume the layer-0 input address them as windows (row b + t)
__global__ void chunk_prep_kernel(WindowSrc w, bf16_t* __restrict__ hi, bf16_t* __restrict__ lo, int64_t rows, int F) {
    const int64_t total = rows * F;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int f = (int)(i % F);
        float v = w.src[(w.start + i / F) * F + f];
        if (w.xmin) v = (v - w.xmin[f]) / (w.xmax[f] - w.xmin[f]);
        const bf16_t h = __float2bfloat16(v);
        hi[i] = h;
        if (lo) lo[i] = __float2bfloat16(v - __bfloat162float(h));
    }
}
// whether a windowed (never collated) layer-0 input is possible: no input dropout to apply, and every GEMM tile of 128
// (64) logical rows stays inside one time step
static inline bool windows_direct(const bigru_plan& p, bool have_windows, bool do_drop) {
    return have_windows && !do_drop && p.B % 128 == 0 && p.F % 8 == 0;
}

// inter-layer dropout: Yrow -> Xrow (masked); rows x cols = R x DH
__global__ void dropout_rows_kernel(const bf16_t* __restrict__ Y, bf16_t* __restrict__ Xrow, int64_t R, int cols, int B, int T,
                                    float pdrop, uint64_t seed, uint32_t stream) {
    const float scale = 1.f / (1.f - pdrop);
    const int64_t total = R * cols;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int cidx = i % cols;
        const int64_t r = i / cols;
        const int64_t b = r % B, t = r / B;
        const uint64_t key = ((uint64_t)b * T + t) * cols + cidx;          // batch-major key, as the fp32 path
        const float v = bigru_uniform(seed, stream, key) < pdrop ? 0.f : __bfloat162float(Y[i]) * scale;
        Xrow[i] = __float2bfloat16(v);
    }
}
// gradient of the same dropout, in place on the BLOCKED fp32 gradient [d][tile][t][cta][thread][8] (see tc_gemm.cuh)
__global__ void dropout_grad_rows_kernel(float* __restrict__ dYB, int64_t R, int cols, int B, int T, int H, float pdrop,
                                         uint64_t seed, uint32_t stream, int wide) {
    const float scale = 1.f / (1.f - pdrop);
    const int64_t total = R * cols;
    const int U = wide ? 64 : 128, NBt = wide ? 32 : 16;          // units per CTA, batch rows per tile (tc_scan.cuh / tc_scan_w.cuh)
    const int CS = H / U, ntl = B / NBt;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int i8 = i & 7;
        int64_t e = i >> 3;
        const int tid = e % 256; e /= 256;
        const int c = e % CS; e /= CS;
        const int t = e % T; e /= T;
        const int tile = e % ntl;
        const int d = e / ntl;
        const int unit = wide ? c * 64 + (tid & 63) : c * 128 + ((tid >> 5) & 3) * 32 + (tid & 31);
        const int64_t b = wide ? tile * 32 + (tid >> 6) * 8 + i8 : tile * 16 + (tid >> 7) * 8 + i8;
        const uint64_t key = ((uint64_t)b * T + t) * cols + (uint64_t)(d * H + unit);
        dYB[i] = bigru_uniform(seed, stream, key) < pdrop ? 0.f : dYB[i] * scale;
    }
}

// W_ih fp32 [3H][I] of direction d -> Wih bf16 rows d*3H.. of [D*3H][I] and WihT bf16 [I][D*3H]
__global__ void pack_wih_kernel(const float* __restrict__ w, bf16_t* __restrict__ Wih, bf16_t* __restrict__ WihT,
                                int H3, int I, int d, int D) {
    const int64_t total = (int64_t)H3 * I;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int k = i % I, q = i / I;
        const bf16_t v = __float2bfloat16(w[i]);
        Wih[((int64_t)d * H3 + q) * I + k] = v;
        WihT[(int64_t)k * D * H3 + (int64_t)d * H3 + q] = v;
    }
}
// bias_fold[d*3H + q] = b_ih[q] + (q < 2H ? b_hh[q] : 0);  b_hn[d*H + j] = b_hh[2H + j]
__global__ void pack_bias_kernel(const float* __restrict__ b_ih, const float* __restrict__ b_hh, float* __restrict__ bfold,
                                 float* __restrict__ bhn, int H, int d) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= 3 * H) return;
    bfold[d * 3 * H + q] = b_ih[q] + (q < 2 * H ? b_hh[q] : 0.f);
    if (q >= 2 * H) bhn[d * H + q - 2 * H] = b_hh[q];
}

// All weight packing of a forward call in ONE launch: blockIdx.y enumerates (layer, direction).
struct PackJob { const float* w_ih; const float* w_hh; const float* b_ih; const float* b_hh;
                 bf16_t* Wih; bf16_t* WihT; bf16_t* Wimg; bf16_t* WTimg; float* bfold; float* bhn; int I; int d; };   // Wih rows hold pad8(I) columns
struct PackJobs { PackJob j[32]; };
// dst_rm[r][c] = dst_t[c][r] = bf16(src[r][c]) for a [rows][cols] fp32 matrix (cols % 32 == 0, rows % 32 == 0): 32 x 32 tiles
// through shared memory so that the row-major AND the transposed image are both written coalesced.  ld_rm / ld_t are the
// leading dimensions of the two images (elements).
__device__ __forceinline__ void pack_tile_pair(const float* __restrict__ src, int rows, int cols, bf16_t* __restrict__ dst_rm, int64_t ld_rm,
                                               bf16_t* __restrict__ dst_t, int64_t ld_t, int tile0, int tile_stride, float (*tile)[33]) {
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;          // 256 threads: 32 x 8
    const int tr = rows / 32, tcn = cols / 32;
    for (int tl = tile0; tl < tr * tcn; tl += tile_stride) {
        const int r0 = (tl / tcn) * 32, c0 = (tl % tcn) * 32;
#pragma unroll
        for (int i = ty; i < 32; i += 8) {
            const float v = src[(int64_t)(r0 + i) * cols + c0 + tx];
            tile[i][tx] = v;
            dst_rm[(int64_t)(r0 + i) * ld_rm + c0 + tx] = __float2bfloat16(v);
        }
        __syncthreads();
#pragma unroll
        for (int i = ty; i < 32; i += 8) dst_t[(int64_t)(c0 + i) * ld_t + r0 + tx] = __float2bfloat16(tile[tx][i]);
        __syncthreads();
    }
}
__global__ void __launch_bounds__(256) pack_all_kernel(const PackJobs jobs, int H, int D) {
    __shared__ float tile[32][33];
    const PackJob& J = jobs.j[blockIdx.y];
    const int H3 = 3 * H, I = J.I, d = J.d;
    if (I % 32 == 0) {
        // W_ih [3H][I] -> rows d*3H.. of Wih [D*3H][I] and columns d*3H.. of WihT [I][D*3H]
        pack_tile_pair(J.w_ih, H3, I, J.Wih + (int64_t)d * H3 * I, I, J.WihT + (int64_t)d * H3, (int64_t)D * H3, blockIdx.x, gridDim.x, tile);
    } else {
        const int Ip = (I + 7) & ~7;                           // zero columns up to the padded row pitch
        const int64_t n_ih = (int64_t)H3 * Ip;
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_ih; i += (int64_t)gridDim.x * blockDim.x) {
            const int k = i % Ip, q = i / Ip;
            const bf16_t v = __float2bfloat16(k < I ? J.w_ih[(int64_t)q * I + k] : 0.f);
            J.Wih[((int64_t)d * H3 + q) * Ip + k] = v;
            if (k < I) J.WihT[(int64_t)k * D * H3 + (int64_t)d * H3 + q] = v;
        }
    }
    // W_hh [3H][H]: gate g of unit u -> Wimg [unit][g][H] (row g*H+u of W_hh is row u*3+g of the image) and W_hh^T
    // -> WTimg [H][3H]; one gate block ([H][H]) at a time so that the row-major image is a plain strided copy
    if (H <= 256)                                           // H = 512: pack_wide_images_kernel (tc_scan_w.cuh) writes the images
        for (int g = 0; g < 3; ++g)
            pack_tile_pair(J.w_hh + (int64_t)g * H * H, H, H, J.Wimg + (int64_t)g * H, (int64_t)3 * H, J.WTimg + (int64_t)g * H, H3,
                           blockIdx.x, gridDim.x, tile);
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < H3; q += (int64_t)gridDim.x * blockDim.x) {
        J.bfold[d * H3 + q] = J.b_ih[q] + (q < 2 * H ? J.b_hh[q] : 0.f);
        if (q >= 2 * H) J.bhn[d * H + q - 2 * H] = J.b_hh[q];
    }
}

// Head forward (biGRU_model.py:111-137) fused: direction sum, last hidden, max / mean pooling over T and the
// Linear(3H -> C), one block (256 threads) per batch row.  Pooling: a thread owns 8 consecutive hidden units (one 16-byte
// load per direction and time step), H/8 lanes cover a time step and the 256/(H/8) lane groups split the T steps; the
// groups' partial (max, first argmax, sum) are combined through shared memory.  H % 8 == 0, H <= 256.
__global__ void __launch_bounds__(256) head_fwd_kernel(const bf16_t* __restrict__ Y, const bf16_t* __restrict__ Ylo, const float* __restrict__ lin_w,
                                                       const float* __restrict__ lin_b, float* __restrict__ cat, int* __restrict__ arg,
                                                       float* __restrict__ logits, int B, int T, int H, int D, int C) {
    extern __shared__ float hs[];                      // [G][H] max, [G][H] sum, [G][H] argmax (int), then [C][8] partial logits
    const int b = blockIdx.x, tid = threadIdx.x;
    const int ld = D * H, LPS = H >> 3, G = 256 / LPS;  // lanes per step, lane groups
    const int grp = tid / LPS, u0 = (tid % LPS) * 8;
    float* s_max = hs; float* s_sum = hs + G * H; int* s_arg = reinterpret_cast<int*>(hs + 2 * G * H);
    float* red = hs + 3 * G * H;
    float mx[8], sm[8]; int am[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { mx[i] = -INFINITY; sm[i] = 0.f; am[i] = 0; }
    if (grp < G) {
#pragma unroll 4
        for (int t = grp; t < T; t += G) {
            const bf16_t* y = Y + ((int64_t)t * B + b) * ld + u0;
            const uint4 a = *reinterpret_cast<const uint4*>(y);
            uint4 c = make_uint4(0u, 0u, 0u, 0u);
            if (D == 2) c = *reinterpret_cast<const uint4*>(y + H);
            const bf16_t* pa = reinterpret_cast<const bf16_t*>(&a);
            const bf16_t* pc = reinterpret_cast<const bf16_t*>(&c);
            uint4 al = make_uint4(0u, 0u, 0u, 0u), cl = al;
            if (Ylo) {
                const bf16_t* yl = Ylo + ((int64_t)t * B + b) * ld + u0;
                al = *reinterpret_cast<const uint4*>(yl);
                if (D == 2) cl = *reinterpret_cast<const uint4*>(yl + H);
            }
            const bf16_t* pal = reinterpret_cast<const bf16_t*>(&al);
            const bf16_t* pcl = reinterpret_cast<const bf16_t*>(&cl);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float v = (__bfloat162float(pa[i]) + __bfloat162float(pal[i])) + (__bfloat162float(pc[i]) + __bfloat162float(pcl[i]));
                if (v > mx[i]) { mx[i] = v; am[i] = t; }
                sm[i] += v;
            }
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) { s_max[grp * H + u0 + i] = mx[i]; s_sum[grp * H + u0 + i] = sm[i]; s_arg[grp * H + u0 + i] = am[i]; }
    }
    __syncthreads();
    // second phase: thread -> units tid, tid + 256 (H <= 512)
    float last2[2] = {0.f, 0.f}, m2[2] = {0.f, 0.f}, avg2[2] = {0.f, 0.f};
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const int j = tid + 256 * k;
        if (j >= H) continue;
        float last = __bfloat162float(Y[((int64_t)(T - 1) * B + b) * ld + j]), m = -INFINITY, sum = 0.f;
        int a_t = 0;
        if (Ylo) last += __bfloat162float(Ylo[((int64_t)(T - 1) * B + b) * ld + j]);
        if (D == 2) {
            float lr = __bfloat162float(Y[(int64_t)b * ld + H + j]);
            if (Ylo) lr += __bfloat162float(Ylo[(int64_t)b * ld + H + j]);
            last += lr;
        }
        for (int g = 0; g < G; ++g) {                  // first occurrence of the maximum, as a sequential scan over t finds it
            const float v = s_max[g * H + j]; const int at = s_arg[g * H + j];
            if (v > m || (v == m && at < a_t)) { m = v; a_t = at; }
            sum += s_sum[g * H + j];
        }
        float* c = cat + (int64_t)b * 3 * H;
        c[j] = last; c[H + j] = m; c[2 * H + j] = sum / (float)T;
        arg[(int64_t)b * H + j] = a_t;
        last2[k] = last; m2[k] = m; avg2[k] = sum / (float)T;
    }
    const int j = tid;
    for (int cc = 0; cc < C; ++cc) {
        float v = 0.f;
        const float* w = lin_w + (int64_t)cc * 3 * H;
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const int jj = tid + 256 * k;
            if (jj < H) v += last2[k] * w[jj] + m2[k] * w[H + jj] + avg2[k] * w[2 * H + jj];
        }
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if ((j & 31) == 0) red[cc * 8 + (j >> 5)] = v;
    }
    __syncthreads();
    for (int cc = j; cc < C; cc += 256) {                 // output_size may exceed the block size
        float v = lin_b[cc];
        for (int w = 0; w < 8; ++w) v += red[cc * 8 + w];
        logits[(int64_t)b * C + cc] = v;
    }
}
// d(lin_w)[c][k] = sum_b dlogits[b][c] cat[b][k];  d(lin_b)[c] = sum_b dlogits[b][c]   (outputs pre-zeroed; the batch
// is split over blockIdx.z and combined with atomics so that the tiny reduction is not one long serial loop)
__global__ void head_bwd_w_kernel(const float* __restrict__ dlogits, const float* __restrict__ cat, float* __restrict__ dlin_w,
                                  float* __restrict__ dlin_b, int B, int H3, int C, int bchunk) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    const int cc = blockIdx.y;
    if (k >= H3) return;
    const int b0 = blockIdx.z * bchunk, b1 = min(B, b0 + bchunk);
    float acc = 0.f, accb = 0.f;
#pragma unroll 4
    for (int b = b0; b < b1; ++b) {
        const float g = dlogits[(int64_t)b * C + cc];
        acc = fmaf(g, cat[(int64_t)b * H3 + k], acc);
        accb += g;
    }
    atomicAdd(dlin_w + (int64_t)cc * H3 + k, acc);
    if (k == 0) atomicAdd(dlin_b + cc, accb);
}

// dW_hh[d] += dgh_first^T h0[d]: the first forward step's h_prev is the caller's initial state, which the time-shifted
// Y operand of the dW_hh GEMM does not contain (it reads zeros there).  dgh = [da_r | da_z] (dgi rows) and da_n * r (dghn rows),
// bf16; the bf16x3 path passes the residual parts as well (dgh = hi + lo), this path passes lo = nullptr.
// Thread = gate row q x DWHH_H0_COLS consecutive columns (one dgh load feeds that many FMAs); grid ((3H+127)/128, H/DWHH_H0_COLS, D).
constexpr int DWHH_H0_COLS = 8;                               // H % 8 == 0 on the tensor-core paths
__global__ void dwhh_h0_kernel(const bf16_t* __restrict__ dgi_hi, const bf16_t* __restrict__ dgi_lo, const bf16_t* __restrict__ dghn_hi,
                               const bf16_t* __restrict__ dghn_lo, const float* __restrict__ h0, float* __restrict__ dwhh, int64_t dir_stride,
                               int B, int T, int H, int D) {
    const int d = blockIdx.z;
    const int q = blockIdx.x * blockDim.x + threadIdx.x;      // gate row of W_hh (0..3H)
    const int k0 = blockIdx.y * DWHH_H0_COLS;                 // first column of W_hh
    if (q >= 3 * H) return;
    const int64_t t_first = d == 0 ? 0 : T - 1;
    float acc[DWHH_H0_COLS];
#pragma unroll
    for (int j = 0; j < DWHH_H0_COLS; ++j) acc[j] = 0.f;
    for (int b = 0; b < B; ++b) {
        const int64_t row = t_first * B + b;
        float g;
        if (q < 2 * H) {
            const int64_t i = row * D * 3 * H + d * 3 * H + q;
            g = dgi_lo ? __bfloat162float(dgi_hi[i]) + __bfloat162float(dgi_lo[i]) : __bfloat162float(dgi_hi[i]);
        } else {
            const int64_t i = row * D * H + d * H + q - 2 * H;
            g = dghn_lo ? __bfloat162float(dghn_hi[i]) + __bfloat162float(dghn_lo[i]) : __bfloat162float(dghn_hi[i]);
        }
        const float* hb = h0 + ((int64_t)d * B + b) * H + k0;
#pragma unroll
        for (int j = 0; j < DWHH_H0_COLS; ++j) acc[j] = fmaf(g, hb[j], acc[j]);
    }
    float* w = dwhh + (int64_t)d * dir_stride + (int64_t)q * H + k0;
#pragma unroll
    for (int j = 0; j < DWHH_H0_COLS; ++j) w[j] += acc[j];
}

// dX^T of layer 0 (fp32 [F][R]) back to the caller's [B][T][F] (+ input-dropout mask); 32x32 smem transpose
__global__ void dx_to_batch_major_kernel(const float* __restrict__ dXT, float* __restrict__ dx, int B, int T, int F,
                                         float pdrop, int spatial, uint64_t seed) {
    __shared__ float tile[32][33];
    const int t = blockIdx.z, b0 = blockIdx.y * 32, f0 = blockIdx.x * 32;
    const int64_t R = (int64_t)T * B;
    const float scale = pdrop > 0.f ? 1.f / (1.f - pdrop) : 1.f;
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        const int f = f0 + i, b = b0 + threadIdx.x;
        tile[i][threadIdx.x] = (b < B && f < F) ? dXT[(int64_t)f * R + (int64_t)t * B + b] : 0.f;
    }
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        const int b = b0 + i, f = f0 + threadIdx.x;
        if (b < B && f < F) {
            float v = tile[threadIdx.x][i];
            if (pdrop > 0.f) {
                const uint64_t key = spatial ? (uint64_t)b * F + f : ((uint64_t)b * T + t) * F + f;
                v = bigru_uniform(seed, 0u, key) < pdrop ? 0.f : v * scale;
            }
            dx[((int64_t)b * T + t) * F + f] = v;
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// GEMM helper with accounting
// ---------------------------------------------------------------------------------------------------
// A / B operand descriptions: K-major [rows][K] (ld = row stride) or MN-major [K rows][MN] (p.a_mn / p.b_mn set)
static int tc_gemm(const void* A, int64_t a_rows, int64_t lda, const void* Bm, int64_t b_rows, int64_t ldb,
                   tcg::Params& p, cudaStream_t st, int kclass = KC_TC_GEMM, const void* Alo = nullptr, const void* Blo = nullptr) {
    CUtensorMap tA, tB, tAl, tBl;
    const bool split = Alo != nullptr && Blo != nullptr;
    p.nsplit = split ? 3 : 1;
    if (split) {
        const int e1 = p.a_mn ? tcg::make_operand_map_mn(&tAl, Alo, (uint64_t)p.K, (uint64_t)a_rows, (uint64_t)lda)
                              : tcg::make_operand_map(&tAl, Alo, (uint64_t)a_rows, (uint64_t)p.K, (uint64_t)lda);
        const int e2 = p.b_mn ? tcg::make_operand_map_mn(&tBl, Blo, (uint64_t)(p.b_win ? p.b_win_rows : p.K), (uint64_t)b_rows, (uint64_t)ldb)
                              : tcg::make_operand_map(&tBl, Blo, (uint64_t)b_rows, (uint64_t)p.K, (uint64_t)ldb);
        if (e1 || e2) { bigru_set_error("cuTensorMapEncodeTiled failed (low operand parts)"); return BIGRU_ERR_CUDA; }
    }
    const int ea = p.a_mn ? tcg::make_operand_map_mn(&tA, A, (uint64_t)p.K, (uint64_t)a_rows, (uint64_t)lda)
                          : tcg::make_operand_map(&tA, A, (uint64_t)a_rows, (uint64_t)p.K, (uint64_t)lda);
    const int eb = p.b_mn ? tcg::make_operand_map_mn(&tB, Bm, (uint64_t)(p.b_win ? p.b_win_rows : p.K), (uint64_t)b_rows, (uint64_t)ldb)
                          : tcg::make_operand_map(&tB, Bm, (uint64_t)b_rows, (uint64_t)p.K, (uint64_t)ldb);
    if (ea || eb) {
        bigru_set_error("cuTensorMapEncodeTiled failed (rows %lld/%lld K %d ld %lld/%lld)", (long long)a_rows,
                        (long long)b_rows, p.K, (long long)lda, (long long)ldb);
        return BIGRU_ERR_CUDA;
    }
    ProfScope ps(kclass, 2.0 * p.M * p.N * (double)p.K * p.batch, 0.0, st);
    CUDA_TRY(tcg::launch(tA, tB, p, st, split ? &tAl : nullptr, split ? &tBl : nullptr));
    return BIGRU_OK;
}

static inline unsigned nblk2(int64_t n, int bs) { return (unsigned)cdiv64(n, bs); }

// ---------------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------------
static int forward_bf16(const bigru_plan& p, const float* params, const float* x, const float* h0, float drop,
                        int spatial, int training, uint64_t seed, void* stash_v, void* scratch_v, float* logits,
                        float* hn, cudaStream_t st, WindowSrc win = WindowSrc{nullptr, nullptr, nullptr, 0}) {
    const Bf16Layout L = bf16_layout(p);
    const bool wide = bf16_wide(p);
    uint8_t* S = (uint8_t*)stash_v;
    uint8_t* W = (uint8_t*)scratch_v;
    const int B = p.B, T = p.T, H = p.H, D = p.D, F = p.F;
    const int64_t R = (int64_t)B * T;
    const bool do_drop = training && drop > 0.f;
    unsigned int* dbg = (unsigned int*)(S + L.dbg);
    CUDA_TRY(cudaMemsetAsync(dbg, 0, 64, st));

    // 1. pack weights to bf16 operand images (one launch for all layers and directions)
    {
        PackJobs jobs{};
        int nj = 0;
        for (int l = 0; l < p.L; ++l)
            for (int d = 0; d < D; ++d) {
                PackJob& J = jobs.j[nj++];
                J.w_ih = params + p.off_wih(l, d); J.w_hh = params + p.off_whh(l, d);
                J.b_ih = params + p.off_bih(l, d); J.b_hh = params + p.off_bhh(l, d);
                J.Wih = (bf16_t*)(S + L.Wih[l]); J.WihT = (bf16_t*)(S + L.WihT[l]);
                J.Wimg = (bf16_t*)(S + L.Wimg[l]) + (size_t)d * 3 * H * H; J.WTimg = (bf16_t*)(S + L.WTimg[l]) + (size_t)d * 3 * H * H;
                J.bfold = (float*)(S + L.bfold[l]); J.bhn = (float*)(S + L.bhn[l]); J.I = (int)p.in_size(l); J.d = d;
            }
        KLAUNCH(KC_PACK, 0.0, 0.0, st, pack_all_kernel<<<dim3(148, nj), 256, 0, st>>>(jobs, H, D));
        if (wide) {
            using WG = tcw::Geo<512>;
            const size_t fimg = (size_t)WG::CS * 128 * WG::ROW_ELEMS, ftail = (size_t)WG::CS * WG::NTAIL * 128 * 64, bimg = (size_t)WG::CS * 128 * WG::NRB * 192;
            for (int l = 0; l < p.L; ++l)
                for (int d = 0; d < D; ++d)
                    KLAUNCH(KC_PACK, 0.0, 0.0, st, tcw::pack_wide_images_kernel<512><<<148 * 2, 256, 0, st>>>(
                                params + p.off_whh(l, d), (bf16_t*)(S + L.Wimg[l]) + d * fimg, (bf16_t*)(S + L.Wimg[l]) + D * fimg + d * ftail,
                                (bf16_t*)(S + L.WTimg[l]) + d * bimg));
        }
    }
    // 2. layer-0 input: cast to bf16, time-major rows (+ input dropout) - or, for windows of a chunk, only the chunk itself
    const bool direct = windows_direct(p, win.src != nullptr, do_drop);
    if (direct)
        KLAUNCH(KC_PACK, 0.0, 6.0 * (B + T - 1) * F, st, chunk_prep_kernel<<<148, 256, 0, st>>>(win, (bf16_t*)(S + L.Xrow[0]), nullptr, (int64_t)B + T - 1, F));
    else if (F % 8 == 0)
        KLAUNCH(KC_PACK, 0.0, 6.0 * R * F, st, cast_x_kernel<<<148 * 8, 256, 0, st>>>(x, win, (bf16_t*)(S + L.Xrow[0]), nullptr, B, T, F,
                                                                                       do_drop ? drop : 0.f, spatial, seed));
    else
        KLAUNCH(KC_PACK, 0.0, 6.0 * R * F, st, cast_x_pad_kernel<<<148 * 8, 256, 0, st>>>(x, win, (bf16_t*)(S + L.Xrow[0]), nullptr, B, T, F, pad8(F),
                                                                                           do_drop ? drop : 0.f, spatial, seed));
    for (int l = 0; l < p.L; ++l) {
        const int I = (int)p.in_size(l);
        const bf16_t* Xrow = (const bf16_t*)(S + L.Xrow[l]);
        if (l > 0) {
            if (do_drop) {
                KLAUNCH(KC_MISC, 0.0, 0.0, st, dropout_rows_kernel<<<148 * 8, 256, 0, st>>>(
                                                   (const bf16_t*)(S + L.Yrow[l - 1]), (bf16_t*)(S + L.Xrow[l]), R, I, B, T,
                                                   drop, seed, (uint32_t)l));
            } else {
                Xrow = (const bf16_t*)(S + L.Yrow[l - 1]);
            }
        }
        // 3. input projection for all t, both directions, written in the scan kernel's blocked layout:  W_ih X^T + bias(row).
        //    With 64 input features (layer 0 of the reference configurations) the projection is formed inside the scan
        //    kernel instead (tc_scan.cuh, fuse_x): no gi round trip through HBM and no GEMM launch.
        const bool fuse_x = (I == 64) && !wide;
        if (!fuse_x) {
            tcg::Params g{};
            const int Ip = pad8(I);                                                     // zero-padded K extent (layer 0, n_features % 8 != 0)
            g.M = D * 3 * H; g.N = (int)R; g.K = Ip; g.batch = 1; g.splitk = 1; g.mode = tcg::OUT_SCAN_BF16;
            g.blk = wide ? tcg::ScanBlk{T, B, H, 3, 64, 32} : tcg::ScanBlk{T, B, H, 3}; g.m_fast = 1;      // the few weight m-tiles share each activation tile via L2
            g.C = W + L.gi; g.ldc = R; g.bias = (const float*)(S + L.bfold[l]); g.bias_per_row = 1; g.dbg = dbg;
            const bool wnd = direct && l == 0;
            g.b_win = wnd ? B : 0;
            TRY(tc_gemm(S + L.Wih[l], D * 3 * H, Ip, Xrow, wnd ? (int64_t)B + T - 1 : R, Ip, g, st));
        }
        // 4. recurrence.  With an initial state its recurrent product W_hh h0 is formed here in fp32 (tiny: B x 3H x H per
        //    direction, no bias) and read by the scan at step 0, which issues no recurrent MMA.
        const float* h0l = h0 ? h0 + (int64_t)l * D * B * H : nullptr;
        if (h0l) {
            GemmArgs r = gemm_args(h0l, params + p.off_whh(l, 0), (float*)(W + L.gh0), B, 3 * H, H, H, 1, H, 1, 3 * H);
            r.batch = D; r.zA = (int64_t)B * H; r.zB = p.ld_block(l); r.zC = (int64_t)B * 3 * H;
            TRY(sgemm_launch(r, st));
        }
        if (wide) {
            using WG = tcw::Geo<512>;
            tcw::FwdParams f{};
            f.B = B; f.T = T; f.H = H; f.D = D;
            f.Wimg = (const bf16_t*)(S + L.Wimg[l]); f.Wtail = f.Wimg + (size_t)D * WG::CS * 128 * WG::ROW_ELEMS;
            f.giW = (const bf16_t*)(W + L.gi); f.b_hn = (const float*)(S + L.bhn[l]);
            f.Yrow = (bf16_t*)(S + L.Yrow[l]); f.GW = (bf16_t*)(S + L.G[l]); f.YBW = (bf16_t*)(S + L.YB[l]);
            f.hn_out = hn ? hn + (int64_t)l * D * B * H : nullptr; f.dbg = dbg;
            f.h0 = h0l; f.gh0 = h0l ? (const float*)(W + L.gh0) : nullptr;
            ProfScope ps(KC_TC_SCAN_FWD, 2.0 * 3 * H * H * (double)R * D, 0.0, st);
            CUDA_TRY(tcw::launch_fwd(f, st));
            continue;
        }
        tcs::FwdParams f{};
        f.B = B; f.T = T; f.H = H; f.D = D;
        f.Wimg = (const bf16_t*)(S + L.Wimg[l]); f.giB = (const bf16_t*)(W + L.gi); f.b_hn = (const float*)(S + L.bhn[l]);
        f.Yrow = (bf16_t*)(S + L.Yrow[l]); f.G = (bf16_t*)(S + L.G[l]); f.YB = (bf16_t*)(S + L.YB[l]);
        f.hn_out = hn ? hn + (int64_t)l * D * B * H : nullptr; f.dbg = dbg;
        f.h0 = h0l; f.gh0 = h0l ? (const float*)(W + L.gh0) : nullptr;
        f.fuse_x = fuse_x ? 1 : 0; f.x_win = (direct && l == 0) ? 1 : 0; f.Xrow = Xrow; f.Wih = (const bf16_t*)(S + L.Wih[l]); f.bfold = (const float*)(S + L.bfold[l]);
        {
            ProfScope ps(KC_TC_SCAN_FWD, 2.0 * 3 * H * H * (double)R * D, 0.0, st);
            CUDA_TRY(tcs::launch_fwd(f, st));
        }
    }
    // 5. head: pooling + Linear fused
    {
        const int G = 256 / (H / 8);
        const size_t hsm = sizeof(float) * ((size_t)3 * G * H + (size_t)p.C * 8);
        KLAUNCH(KC_HEAD, 0.0, 2.0 * R * D * H, st, head_fwd_kernel<<<B, 256, hsm, st>>>(
                    (const bf16_t*)(S + L.Yrow[p.L - 1]), nullptr, params + p.off_linw(), params + p.off_linb(), (float*)(S + L.cat),
                    (int*)(S + L.arg), logits, B, T, H, D, p.C));
    }
    return BIGRU_OK;
}

// ---------------------------------------------------------------------------------------------------
// backward
// ---------------------------------------------------------------------------------------------------
static int backward_bf16(const bigru_plan& p, const float* params, const float* x, const float* h0, float drop,
                         int spatial, int training, uint64_t seed, const void* stash_v, void* scratch_v,
                         const float* dlogits, float* grads, float* dx, float* dh0, cudaStream_t st, int l_from = -1, int l_to = 0) {
    // layers l_from .. l_to (downwards; l_from = -1: from the top layer).  A call that starts at the top layer also zeroes the gradient
    // vector and forms the head's gradients; a later call for the lower layers continues from the dY the upper call left in scratch.
    if (l_from < 0) l_from = p.L - 1;
    const bool from_top = l_from == p.L - 1;
    const Bf16Layout L = bf16_layout(p);
    const bool wide = bf16_wide(p);
    const uint8_t* S = (const uint8_t*)stash_v;
    uint8_t* W = (uint8_t*)scratch_v;
    const int B = p.B, T = p.T, H = p.H, D = p.D, C = p.C;
    const int64_t R = (int64_t)B * T;
    const bool do_drop = training && drop > 0.f;
    unsigned int* dbg = (unsigned int*)(const_cast<uint8_t*>(S) + L.dbg);
    if (from_top) CUDA_TRY(cudaMemsetAsync(grads, 0, sizeof(float) * p.nparams, st));
    const float* cat = (const float*)(S + L.cat);
    if (from_top) {
        const int bchunk = 16;
        KLAUNCH(KC_HEAD, 0.0, 0.0, st, head_bwd_w_kernel<<<dim3(nblk2(3 * H, 128), C, (B + bchunk - 1) / bchunk), 128, 0, st>>>(
                    dlogits, cat, grads + p.off_linw(), grads + p.off_linb(), B, 3 * H, C, bchunk));
    }
    float* dY = (float*)(W + L.dYa);
    float* dYnext = (float*)(W + L.dYb);
    if ((p.L - 1 - l_from) & 1) { float* t_ = dY; dY = dYnext; dYnext = t_; }      // the buffers alternate per layer
    for (int l = l_from; l >= l_to; --l) {
        const int I = (int)p.in_size(l);
        const float* h0l = h0 ? h0 + (int64_t)l * D * B * H : nullptr;
        float* dh0l = dh0 ? dh0 + (int64_t)l * D * B * H : nullptr;
        // 1. BPTT scan
        if (wide) {
            tcw::BwdParams b{};
            b.B = B; b.T = T; b.H = H; b.D = D;
            b.WTimg = (const bf16_t*)(S + L.WTimg[l]); b.GW = (const bf16_t*)(S + L.G[l]); b.YBW = (const bf16_t*)(S + L.YB[l]);
            b.dYBW = dY; b.h0 = h0l; b.dh0 = dh0l;
            if (l == p.L - 1) { b.dlogits = dlogits; b.lin_w = params + p.off_linw(); b.arg = (const int*)(S + L.arg); b.C = C; }
            b.dgi_row = (bf16_t*)(W + L.gi); b.dghn_row = (bf16_t*)(W + L.dghn);
            b.db_ih = grads + p.off_bih(l, 0); b.db_hh = grads + p.off_bhh(l, 0); b.dir_stride = p.ld_block(l); b.dbg = dbg;
            ProfScope ps(KC_TC_SCAN_BWD, 2.0 * 3 * H * H * (double)R * D, 0.0, st);
            CUDA_TRY(tcw::launch_bwd(b, st));
        } else {
            tcs::BwdParams b{};
            b.B = B; b.T = T; b.H = H; b.D = D;
            b.WTimg = (const bf16_t*)(S + L.WTimg[l]); b.G = (const bf16_t*)(S + L.G[l]); b.YB = (const bf16_t*)(S + L.YB[l]);
            b.dYB = dY; b.h0 = h0l; b.dh0 = dh0l;
            if (l == p.L - 1) { b.dlogits = dlogits; b.lin_w = params + p.off_linw(); b.arg = (const int*)(S + L.arg); b.C = C; }
            b.dgi_row = (bf16_t*)(W + L.gi); b.dghn_row = (bf16_t*)(W + L.dghn);
            b.db_ih = grads + p.off_bih(l, 0); b.db_hh = grads + p.off_bhh(l, 0); b.dir_stride = p.ld_block(l); b.dbg = dbg;
            ProfScope ps(KC_TC_SCAN_BWD, 2.0 * 3 * H * H * (double)R * D, 0.0, st);
            CUDA_TRY(tcs::launch_bwd(b, st));
        }
        // layer input as the projection saw it (row-major, time-major rows)
        const bool dropped = do_drop && (l == 0 || p.L > 1);
        const bf16_t* Xin = (l == 0 || dropped) ? (const bf16_t*)(S + L.Xrow[l]) : (const bf16_t*)(S + L.Yrow[l - 1]);
        // 2. dW_ih[d] = dgi[d]^T X   (M=3H, N=I, K=R): both operands are the row-major activations read MN-major,
        //    both directions in one launch, split-K with TMA reduce-add
        {
            tcg::Params g{};
            g.M = 3 * H; g.N = I; g.K = (int)R; g.batch = D; g.mode = tcg::OUT_ATOMIC_F32; g.a_mn = 1; g.b_mn = 1;
            const int tiles = ((3 * H + 127) / 128) * ((I + 127) / 128) * D;
            g.splitk = (int)std::max<int64_t>(1, std::min<int64_t>((R + 63) / 64, (148 * 2 + tiles / 2) / tiles));    // one full wave at 2 CTAs/SM
            g.C = grads + p.off_wih(l, 0); g.ldc = I; g.zC = p.ld_block(l);
            for (int d = 0; d < D; ++d) { g.a_row_off[d] = d * 3 * H; g.b_row_off[d] = 0; g.b_k_off[d] = 0; }
            g.dbg = dbg;
            g.b_win = (l == 0 && windows_direct(p, x == nullptr, do_drop)) ? B : 0;      // forward_windows left only the chunk in the stash
            g.b_win_rows = B + T - 1;
            TRY(tc_gemm(W + L.gi, (int64_t)D * 3 * H, (int64_t)D * 3 * H, Xin, I, pad8(I), g, st, KC_TC_GEMM_DWIH));   // I columns, padded row pitch
        }
        // 3. dW_hh[d] = dgh[d]^T H_prev  with H_prev(t) = Y(t-1) (dir 0) / Y(t+1) (dir 1): a shift of -+B ROWS of the
        //    time-major output; rows outside [0, R) read as zero through TMA (h_prev = 0 at the first step; an initial state's
        //    term is added by dwhh_h0_kernel below).  dgh = [da_r | da_z] (columns of dgi_row) and da_n*r (dghn_row): two launches.
        for (int part = 0; part < 2; ++part) {
            tcg::Params g{};
            g.M = part == 0 ? 2 * H : H; g.N = H; g.K = (int)R; g.batch = D; g.mode = tcg::OUT_ATOMIC_F32; g.a_mn = 1; g.b_mn = 1;
            const int tiles = ((g.M + 127) / 128) * ((H + 127) / 128) * D;
            g.splitk = (int)std::max<int64_t>(1, std::min<int64_t>((R + 63) / 64, (148 * 2 + tiles / 2) / tiles));
            g.C = grads + p.off_whh(l, 0) + (part == 0 ? 0 : (int64_t)2 * H * H); g.ldc = H; g.zC = p.ld_block(l);
            for (int d = 0; d < D; ++d) {
                g.a_row_off[d] = part == 0 ? d * 3 * H : d * H;
                g.b_row_off[d] = d * H; g.b_k_off[d] = d == 0 ? -B : B;
            }
            g.dbg = dbg;
            if (part == 0) TRY(tc_gemm(W + L.gi, (int64_t)D * 3 * H, (int64_t)D * 3 * H, S + L.Yrow[l], (int64_t)D * H, (int64_t)D * H, g, st, KC_TC_GEMM_DWHH));
            else TRY(tc_gemm(W + L.dghn, (int64_t)D * H, (int64_t)D * H, S + L.Yrow[l], (int64_t)D * H, (int64_t)D * H, g, st, KC_TC_GEMM_DWHH));
        }
        if (h0l)
            KLAUNCH(KC_MISC, 0.0, 0.0, st, dwhh_h0_kernel<<<dim3((3 * H + 127) / 128, H / DWHH_H0_COLS, D), 128, 0, st>>>(
                        (const bf16_t*)(W + L.gi), nullptr, (const bf16_t*)(W + L.dghn), nullptr, h0l, grads + p.off_whh(l, 0), p.ld_block(l),
                        B, T, H, D));
        // 4. dX^T = W_ih^T (both directions concatenated along K = D*3H) x dgi_row^T.  For l > 0 it is written directly in
        //    the blocked layout the next backward scan reads; for layer 0 (caller wants dx) as [F][R] and then re-laid.
        const bool need_dx = l > 0 || dx != nullptr;
        if (need_dx) {
            tcg::Params g{};
            g.M = I; g.N = (int)R; g.K = D * 3 * H; g.batch = 1; g.splitk = 1;
            g.mode = l > 0 ? tcg::OUT_SCAN_F32 : tcg::OUT_F32;
            g.blk = wide ? tcg::ScanBlk{T, B, H, 1, 64, 32} : tcg::ScanBlk{T, B, H, 1}; g.m_fast = 1;
            g.C = dYnext; g.ldc = R; g.dbg = dbg;
            TRY(tc_gemm(S + L.WihT[l], I, (int64_t)D * 3 * H, W + L.gi, R, (int64_t)D * 3 * H, g, st, KC_TC_GEMM_DX));
            if (l > 0 && dropped)
                KLAUNCH(KC_MISC, 0.0, 0.0, st, dropout_grad_rows_kernel<<<148 * 8, 256, 0, st>>>(dYnext, R, I, B, T, H, drop, seed, (uint32_t)l, wide ? 1 : 0));
            if (l == 0) {
                dim3 grid((I + 31) / 32, (B + 31) / 32, T);
                KLAUNCH(KC_MISC, 0.0, 0.0, st, dx_to_batch_major_kernel<<<grid, dim3(32, 8), 0, st>>>(dYnext, dx, B, T, I,
                                                                                               do_drop ? drop : 0.f, spatial, seed));
            }
        }
        float* tmp = dY; dY = dYnext; dYnext = tmp;
    }
    return BIGRU_OK;
}
