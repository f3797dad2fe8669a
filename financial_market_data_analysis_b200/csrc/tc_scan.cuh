// tc_scan.cuh - persistent GRU recurrence on tcgen05 tensor cores (bf16 operands, fp32 accumulate/state).
//
// One thread-block CLUSTER walks all T steps of one (direction, 16-row batch tile).  The cluster has
// CS = H/128 CTAs; CTA c owns hidden units [128c, 128c+128) and keeps its slice of W_hh (3 gates x 128
// rows x H, bf16 = 192 KB at H=256) RESIDENT IN TENSOR MEMORY for the whole scan: the weights are the
// A operand of tcgen05.mma read straight from TMEM (lane = unit row, two bf16 per 32-bit column), so a
// step moves only the 512-byte h slices of the B operand through shared memory.
// Per step ("swap-AB": weights are the M side, the batch tile is the N=16 side):
//     D_g[unit, b] = sum_k W_hg[unit, k] * h_{t-1}[b, k]        g in {r, z, n}   (tcgen05.mma M=128 N=16 K=16)
// accumulators live in TMEM (3 x 16 columns); 8 epilogue warps read them back (tcgen05.ld), add the
// precomputed input projection gi (bf16, bias folded), apply sigmoid/tanh and the state update with the
// fp32 state held in registers, and write the new h (bf16) straight into the UMMA operand tile of the
// next step - locally with st.shared and into every peer CTA with one cp.async.bulk (DSMEM) that
// completes on the peer's mbarrier.  h never goes through HBM on the critical path; what is streamed out
// per step is the layer output (row-major and transposed, for the next layer's GEMMs) and the gate stash.
//
// Layouts (time-major rows r = t*B + b, R = T*B):
// Blocked ("scan-private") layouts: block (d, tile, t, cta) = (((d*ntiles + tile)*T + t)*CS + cta); inside a block
// [gate][thread 0..255][8 batch columns], so a block is one contiguous run that a single cp.async.bulk prefetches
// into a shared-memory ring several steps ahead (per-step HBM latency never sits on the step chain):
//   giB  bf16 [block][3][256][8]   input projection incl. b_ih (+ b_hh for r,z), written by tc_gemm OUT_SCAN_BF16 (read)
//   G    bf16 [block][4][256][8]   r, z, n, hn = W_hn h + b_hn  (stash for backward)              (written)
//   YB   bf16 [block][256][8]      h_t (h_{t-1} of the backward scan)                            (written)
//   Yrow bf16 [R][D*H]    layer output                                        (written)
//   Wimg bf16 [D][H units][3][H]  per-unit rows of W_hh (r|z|n), copied to TMEM   (read once)
#pragma once
#include "tc_common.cuh"

namespace tcs {

#ifdef BIGRU_SCAN_TIMING
#define SCAN_TS(slot) do { if (blockIdx.x == 0 && s >= 64 && s < 72) p.ts[(s - 64) * 16 + (slot)] = clock64(); } while (0)
#else
#define SCAN_TS(slot) do { } while (0)
#endif

constexpr int NB = 16;            // batch rows per tile = UMMA N
constexpr int UNITS = 128;        // hidden units per CTA = UMMA M
constexpr int EPI_WARPS = 8;
constexpr int THREADS = (EPI_WARPS + 2) * 32;    // + MMA/control warp + input-prefetch warp
constexpr int W_CHUNK = UNITS * 128;             // bytes of one [128 x 64] bf16 chunk
constexpr int H_CHUNK = NB * 128;                // bytes of one [16 x 64] bf16 chunk

__device__ __forceinline__ float tanh_fast(float x) { float y; asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float sigmoid_fast(float x) { return fmaf(0.5f, tanh_fast(0.5f * x), 0.5f); }

__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&v)[8]) {
    uint32_t r0, r1, r2, r3, r4, r5, r6, r7;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3), "=r"(r4), "=r"(r5), "=r"(r6), "=r"(r7) : "r"(taddr) : "memory");
    v[0] = __uint_as_float(r0); v[1] = __uint_as_float(r1); v[2] = __uint_as_float(r2); v[3] = __uint_as_float(r3);
    v[4] = __uint_as_float(r4); v[5] = __uint_as_float(r5); v[6] = __uint_as_float(r6); v[7] = __uint_as_float(r7);
}

__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
        ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
          "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]),
          "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]),
          "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31]) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// D[tmem] (+)= A[tmem] * B[smem]: A is read from tensor memory (lane = row, 2 bf16 per column)
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}

// Weight slice -> TMEM.  Wpk holds, per unit row of this CTA, `row_elems` bf16 (the K extent of the A operand);
// the 8 epilogue warps copy it to columns [a_col, a_col + row_elems/2): warp quarter = lane group, warp half =
// column half, 32 columns (64 bf16 = 128 B of the row) per tcgen05.st.
__device__ __forceinline__ void load_weights_to_tmem(const __nv_bfloat16* wrow_base, int row_elems, uint32_t tmem,
                                                     uint32_t a_col, int warp, int lane) {
    const int q = warp & 3, half = warp >> 2;
    const int cols_half = row_elems / 4;                 // columns per half (row_elems/2 columns in total)
    const uint4* src = reinterpret_cast<const uint4*>(wrow_base + (size_t)(q * 32 + lane) * row_elems + (size_t)half * (row_elems / 2));
    for (int i = 0; i < cols_half / 32; ++i) {
        uint32_t v[32];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const uint4 u = src[i * 8 + k];
            v[4 * k] = u.x; v[4 * k + 1] = u.y; v[4 * k + 2] = u.z; v[4 * k + 3] = u.w;
        }
        tmem_st32(tmem + ((uint32_t)(q * 32) << 16) + a_col + (uint32_t)(half * cols_half + i * 32), v);
    }
    tmem_st_wait();
}

// block index of (direction, tile, time step, CTA-in-cluster)
__device__ __forceinline__ size_t blk_index(int d, int tile, int t, int c, int ntiles, int T, int CS) {
    return (((size_t)d * ntiles + tile) * T + t) * CS + c;
}

__device__ __forceinline__ void epi_barrier() { asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory"); }

constexpr int GI_BLOCK = 3 * 256 * 16;    // bytes of one giB block
constexpr int G_BLOCK = 4 * 256 * 16;     // bytes of one stash block
constexpr int YB_BLOCK = 256 * 16;        // bytes of one blocked-h block
constexpr int DY_BLOCK = 256 * 32;        // bytes of one blocked fp32 dY block
constexpr int NSF = 4;                    // forward input ring depth
constexpr int NSB = 3;                    // backward input ring depth
constexpr int BWD_STAGE = G_BLOCK + YB_BLOCK + DY_BLOCK;
constexpr int HEAD_CONST = 3 * 256 * 32;   // top layer: per-thread davg/T, dmax, argmax (8 values each)

constexpr int NSX = 8;                    // fused input projection: x-tile ring depth
constexpr int X_TILE = NB * 128;          // one [16 rows x 64 features] bf16 tile, K-major / 128B swizzle (2 KB)
constexpr int WX_TILE = UNITS * 128;      // n-gate rows of W_ih of this CTA: [128 units x 64 features] (16 KB)
static inline size_t fwd_smem_bytes(int H, bool fuse_x = false) {
    const int KC = H / 64;
    if (fuse_x) return (size_t)2 * KC * H_CHUNK + (size_t)NSX * X_TILE + WX_TILE + 1024 + 256;
    return (size_t)2 * KC * H_CHUNK + (size_t)NSF * GI_BLOCK + 1024 + 256;
}
constexpr uint32_t FWD_A_COL = 64;        // accumulators in columns [0, 64): r, z, W_hn h, (fused: W_in x); weights from column 64
__host__ __device__ static inline uint32_t fwd_tmem_cols(int H, bool fuse_x = false) { return (64 + 3 * H / 2 + (fuse_x ? 64 : 0)) <= 256 ? 256u : 512u; }

struct FwdParams {
    int B, T, H, D;
    const __nv_bfloat16* Wimg;
    const __nv_bfloat16* giB;
    const float* b_hn;            // [D][H]
    __nv_bfloat16* Yrow;          // written by TMA tile stores straight from the h operand tile (tmY)
    __nv_bfloat16* G;
    __nv_bfloat16* YB;
    float* hn_out;                // [D][B][H] fp32, nullable
    const float* h0;              // nullable [D][B][H]: initial hidden state of this layer ...
    const float* gh0;             // ... and its recurrent product W_hh h0 [D][B][3H] (fp32, no bias, formed by the caller): step 0 reads it
    unsigned int* dbg;
    // fused input projection (layer 0, n_features == 64): gi_t = W_ih x_t + b is formed by the same tensor pipe between
    // the recurrent products (it is idle while the epilogue works), giB is not read
    int fuse_x;
    int x_win;                    // 1: Xrow is a chunk [B+T-1][64] and x_t of batch row b is chunk row b + t (zero-copy windows)
    const __nv_bfloat16* Xrow;    // [R][64] time-major input rows
    const __nv_bfloat16* Wih;     // [D*3H][64] (rows r|z|n of direction d at d*3H)
    const float* bfold;           // [D*3H]  b_ih (+ b_hh for r, z)
    CUtensorMap tmY;              // Yrow as [R rows][D*H], box 64 x 16, 128B swizzle (filled by launch_fwd)
    CUtensorMap tmX, tmW;         // fused: Xrow box 64 x 16, Wih box 64 x 128 (filled by launch_fwd)
#ifdef BIGRU_SCAN_TIMING
    unsigned long long* ts;       // bring-up only: clock64 stamps of CTA 0, steps [64, 72), 16 slots per step
#endif
};

// One group of K chunks (NCH x 64 columns of h) of all three gates, fully unrolled: every operand address is a base
// that is fixed for the step plus a compile-time constant, so the 12*NCH tcgen05.mma issue back to back (~9 cycles
// each; a rolled loop with run-time descriptors costs ~26).
template <int H, int NCH, bool FIRST, bool FX = false>
__device__ __forceinline__ void fwd_issue_group(uint32_t tmem_d, uint32_t tmem_a_grp, uint64_t desc_grp) {
    constexpr uint32_t idesc = tc::umma_idesc_bf16(UNITS, NB);
#pragma unroll
    for (int g = 0; g < 3; ++g) {
#pragma unroll
        for (int u = 0; u < NCH; ++u) {
#pragma unroll
            for (int kk = 0; kk < 4; ++kk)       // K = 16 bf16 = 8 TMEM columns of A, 32 B of B
                umma_bf16_ts(tmem_d + (uint32_t)(g * NB), tmem_a_grp + (uint32_t)(g * (H / 2) + (u * 4 + kk) * 8),
                             desc_grp + (uint64_t)(u * (H_CHUNK >> 4) + 2 * kk), idesc,
                             (FIRST && u == 0 && kk == 0 && (!FX || g == 2)) ? 0u : 1u);
        }
    }
}
// fused input projection of one step: D_r, D_z = W_ir x, W_iz x (A in tensor memory, columns xw_col..), D_nx = W_in x
// (A in shared memory: tensor memory is full) - 12 MMAs, all overwrite their accumulators
__device__ __forceinline__ void fwd_issue_x(uint32_t tmem, uint32_t xw_col, uint64_t desc_wn, uint64_t desc_x) {
    constexpr uint32_t idesc = tc::umma_idesc_bf16(UNITS, NB);
#pragma unroll
    for (int g = 0; g < 2; ++g) {
#pragma unroll
        for (int kk = 0; kk < 4; ++kk)
            umma_bf16_ts(tmem + (uint32_t)(g * NB), tmem + xw_col + (uint32_t)(g * 32 + kk * 8), desc_x + (uint64_t)(2 * kk), idesc, kk ? 1u : 0u);
    }
#pragma unroll
    for (int kk = 0; kk < 4; ++kk)
        tc::umma_bf16(tmem + 3 * NB, desc_wn + (uint64_t)(2 * kk), desc_x + (uint64_t)(2 * kk), idesc, kk ? 1u : 0u);
}

template <int H, bool FX>
__global__ void __launch_bounds__(THREADS, 1) gru_scan_fwd_kernel(const __grid_constant__ FwdParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    constexpr int KC = H / 64, CS = H / UNITS, MYCH = UNITS / 64;
    const int B = p.B, T = p.T, D = p.D;
    uint8_t* sH = smem;                                    // [2][KC][H_CHUNK]  h operand tiles
    uint8_t* sIn = sH + (size_t)2 * KC * H_CHUNK;          // [NSF][GI_BLOCK] prefetched gi blocks, or (FX) [NSX][X_TILE] x tiles + W_in tile
    uint8_t* sWn = sIn + (size_t)NSX * X_TILE;             // FX only
    constexpr int NS = FX ? NSX : NSF;
    uint64_t* bars = reinterpret_cast<uint64_t*>(FX ? sWn + WX_TILE : sIn + (size_t)NSF * GI_BLOCK);
    uint64_t* h_full = bars;           // [2]  the peer's h chunk landed (tx bytes of its st.async stores), armed by the control thread
    uint64_t* mma_done = bars + 2;
    uint64_t* acc_free = bars + 3;     // FX: the epilogue has read the accumulators of this step (one arrival per warp)
    uint64_t* w_full = bars + 4;       // FX: W_in tile landed
    uint64_t* epi_done = bars + 5;     // one arrival per epilogue warp: local h chunk written
    uint64_t* in_full = bars + 6;      // [NS]
    uint64_t* in_empty = bars + 6 + NS;    // [NS]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 6 + 2 * NS);
    constexpr uint32_t XW_COL = FWD_A_COL + 3 * H / 2;     // FX: W_ir | W_iz of this CTA's units, 32 columns each

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t c = CS > 1 ? tc::cluster_ctarank() : 0u;
    const int cluster_id = blockIdx.x / CS;
    const int ntiles = B / NB;
    const int d = cluster_id / ntiles, tile = cluster_id % ntiles;
    const int64_t R = (int64_t)T * B;

    if (threadIdx.x == 0) {
        tc::mbar_init(&h_full[0], 1);
        tc::mbar_init(&h_full[1], 1);
        tc::mbar_init(mma_done, 1);
        tc::mbar_init(acc_free, EPI_WARPS);
        tc::mbar_init(w_full, 1);
        tc::mbar_init(epi_done, EPI_WARPS);
        for (int i = 0; i < NS; ++i) { tc::mbar_init(&in_full[i], 1); tc::mbar_init(&in_empty[i], FX ? 1 : EPI_WARPS); }
        tc::fence_mbar_init();
    }
    if (warp == EPI_WARPS) tc::tmem_alloc(tmem_slot, fwd_tmem_cols(H, FX));
    tc::tcgen05_fence_before();
    __syncthreads();
    if (CS > 1) tc::cluster_sync_all();        // every CTA's barriers exist before any peer signals them
    tc::tcgen05_fence_after();
    const uint32_t tmem = *tmem_slot;
    const uint32_t chunk_bytes_mine = (uint32_t)(UNITS / 64) * H_CHUNK;    // the 2 K-chunks this CTA produces
    // W_hh slice of this CTA -> tensor memory (stays there for all T steps)
    if (warp < EPI_WARPS)
        load_weights_to_tmem(p.Wimg + ((size_t)d * CS + c) * UNITS * 3 * H, 3 * H, tmem, FWD_A_COL, warp, lane);
    if (FX && warp < EPI_WARPS) {
        // W_ir (warps 0-3) / W_iz (warps 4-7) rows of this CTA's units -> 32 columns each: lane = unit, 64 bf16 = one tcgen05.st
        const int q = warp & 3, g = warp >> 2;
        const uint4* src = reinterpret_cast<const uint4*>(p.Wih + ((size_t)d * 3 * H + (size_t)g * H + (size_t)c * UNITS + q * 32 + lane) * 64);
        uint32_t v[32];
#pragma unroll
        for (int k = 0; k < 8; ++k) { const uint4 u = src[k]; v[4 * k] = u.x; v[4 * k + 1] = u.y; v[4 * k + 2] = u.z; v[4 * k + 3] = u.w; }
        tmem_st32(tmem + ((uint32_t)(q * 32) << 16) + XW_COL + (uint32_t)(g * 32), v);
        tmem_st_wait();
    }
    tc::tcgen05_fence_before();
    __syncthreads();
    tc::tcgen05_fence_after();

    if (FX && warp == EPI_WARPS + 1) {
        // ---- fused projection: W_in tile once, then one x tile (2 KB, TMA box 64 x 16 -> UMMA K-major layout) per step
        if (tc::elect_one()) {
            bool ok = true;
            tc::mbar_arrive_expect_tx(w_full, WX_TILE);
            tc::tma_load_2d(sWn, &p.tmW, w_full, 0, d * 3 * H + 2 * H + (int)c * UNITS);
            for (int s = 0; s < T; ++s) {
                const int st = s % NSX;
                if (s >= NSX && ok) ok = tc::mbar_wait(&in_empty[st], ((s / NSX) - 1) & 1, p.dbg, 0x300 + (s & 0xff));
                const int t = d == 0 ? s : T - 1 - s;
                tc::mbar_arrive_expect_tx(&in_full[st], X_TILE);
                tc::tma_load_2d(sIn + (size_t)st * X_TILE, &p.tmX, &in_full[st], 0, p.x_win ? t + tile * NB : t * B + tile * NB);
            }
        }
    } else if (warp == EPI_WARPS + 1) {
        // ---- input prefetch: one bulk copy (12 KB) per step into the ring, up to NSF steps ahead
        if (tc::elect_one()) {
            bool ok = true;
            for (int s = 0; s < T; ++s) {
                const int st = s % NSF;
                if (s >= NSF && ok) ok = tc::mbar_wait(&in_empty[st], ((s / NSF) - 1) & 1, p.dbg, 0x300 + (s & 0xff));
                const int t = d == 0 ? s : T - 1 - s;
                tc::mbar_arrive_expect_tx(&in_full[st], GI_BLOCK);
                tc::bulk_g2s(sIn + (size_t)st * GI_BLOCK,
                             reinterpret_cast<const uint8_t*>(p.giB) + blk_index(d, tile, t, (int)c, ntiles, T, CS) * GI_BLOCK,
                             GI_BLOCK, &in_full[st]);
            }
        }
    } else if (warp == EPI_WARPS) {
        // ---- control thread: sequences the step chain.  h_{s-1} is complete when the 8 epilogue warps have
        // written the local chunk (epi_done) and the peers' chunks have landed (h_full, DSMEM bulk copies that
        // this thread also issues for the local chunk); then it issues the 48 MMAs of step s.
        if (tc::elect_one()) {
            bool ok = true;
            if (CS > 1 && T > 1) tc::mbar_arrive_expect_tx(&h_full[0], (uint32_t)(CS - 1) * chunk_bytes_mine);
            auto store_tile = [&](int step) {             // this CTA's 128 columns of Yrow for time step `step`
                const int tt = d == 0 ? step : T - 1 - step;
                const uint8_t* src = sH + (size_t)(step & 1) * KC * H_CHUNK + (size_t)c * chunk_bytes_mine;
                for (int k = 0; k < MYCH; ++k)
                    tc::tma_store_2d(&p.tmY, src + (size_t)k * H_CHUNK, d * H + (int)c * UNITS + 64 * k, tt * B + tile * NB);
                tc::tma_store_commit();
            };
            // per-step operand bases: K chunks [2c, 2c+2) of h_{s-1} are produced by this CTA (local group), the others
            // arrive from the peer over DSMEM (remote group, CS == 2)
            const uint32_t a_loc = tmem + FWD_A_COL + (uint32_t)c * (MYCH * 32);
            const uint32_t a_rem = tmem + FWD_A_COL + (uint32_t)(1 - (int)c) * (MYCH * 32);
            const uint32_t hb0 = tc::smem_u32(sH);
            const uint64_t d_loc0 = tc::umma_desc_k_sw128(hb0 + (uint32_t)c * chunk_bytes_mine);
            const uint64_t d_rem0 = tc::umma_desc_k_sw128(hb0 + (uint32_t)(1 - (int)c) * chunk_bytes_mine);
            constexpr uint64_t BUF_DESC = (uint64_t)((KC * H_CHUNK) >> 4);        // descriptor distance of the two h buffers
            uint64_t desc_wn = 0, desc_x0 = 0;
            if (FX) {
                desc_wn = tc::umma_desc_k_sw128(tc::smem_u32(sWn));
                desc_x0 = tc::umma_desc_k_sw128(tc::smem_u32(sIn));
                if (ok) ok = tc::mbar_wait(w_full, 0, p.dbg, 0xb00);
            }
            for (int s = FX ? 0 : 1; s < T; ++s) {         // after a watchdog hit: keep signalling, stop waiting
                const int pb = (s - 1) & 1;
                if (FX) {
                    // the input projection of step s goes into the accumulators as soon as the epilogue of step s-1 has
                    // read them, and runs while that epilogue does its gate math
                    const int st = s % NSX;
                    if (s > 0 && ok) ok = tc::mbar_wait(acc_free, (s - 1) & 1, p.dbg, 0xc00 + (s & 0xff));
                    if (ok) ok = tc::mbar_wait(&in_full[st], (s / NSX) & 1, p.dbg, 0xd00 + (s & 0xff));
                    tc::tcgen05_fence_after();
                    fwd_issue_x(tmem, XW_COL, desc_wn, desc_x0 + (uint64_t)(st * (X_TILE >> 4)));
                    tc::umma_commit(&in_empty[st]);        // the x tile may be refilled when these MMAs have retired
                    if (s == 0) { tc::umma_commit(mma_done); continue; }      // h_{-1} = 0: no recurrent product
                }
                if (ok) ok = tc::mbar_wait(epi_done, (s - 1) & 1, p.dbg, 0x400 + (s & 0xff));
                SCAN_TS(0);
                tc::tcgen05_fence_after();
                if (CS > 1) {
                    // the local group's MMAs are issued right away and run while the peer's chunks (written straight into
                    // this CTA's operand tile by the peer's epilogue threads) are still in flight
                    fwd_issue_group<H, MYCH, true, FX>(tmem, a_loc, d_loc0 + (pb ? BUF_DESC : 0));
                    SCAN_TS(1);
                    if (ok) ok = tc::mbar_wait(&h_full[pb], ((s - 1) >> 1) & 1, p.dbg, 0x500 + (s & 0xff));
                    SCAN_TS(2);
                    if (s + 1 < T) tc::mbar_arrive_expect_tx(&h_full[s & 1], (uint32_t)(CS - 1) * chunk_bytes_mine);
                    tc::tcgen05_fence_after();
                    fwd_issue_group<H, MYCH, false, FX>(tmem, a_rem, d_rem0 + (pb ? BUF_DESC : 0));
                } else {
                    fwd_issue_group<H, KC, true, FX>(tmem, a_loc, d_loc0 + (pb ? BUF_DESC : 0));
                }
                tc::tma_store_wait_read();                // the tile stored two steps ago is re-written after this commit
                tc::umma_commit(mma_done);
                SCAN_TS(3);
                SCAN_TS(4);
                // layer output rows of step s-1: TMA tile store straight from the operand tile (off the chain)
                store_tile(s - 1);
            }
            if (ok) ok = tc::mbar_wait(epi_done, (T - 1) & 1, p.dbg, 0x400);
            store_tile(T - 1);
            tc::tma_store_wait_all();
        }
    } else if (warp < EPI_WARPS) {
        // ---- epilogue: thread = hidden unit (TMEM lane), 8 of the 16 batch columns
        const int q = warp & 3, half = warp >> 2;
        const int j = q * 32 + lane;
        const int unit = (int)c * UNITS + j;
        const int col0 = half * 8;
        const int tid = threadIdx.x;
        const float bhn = p.b_hn[d * H + unit];
        const float bx_r = FX ? p.bfold[d * 3 * H + unit] : 0.f, bx_z = FX ? p.bfold[d * 3 * H + H + unit] : 0.f,
                    bx_n = FX ? p.bfold[d * 3 * H + 2 * H + unit] : 0.f;
        const bool has_h0 = p.h0 != nullptr && p.gh0 != nullptr;
        float hprev[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) hprev[i] = has_h0 ? p.h0[((int64_t)d * B + tile * NB + col0 + i) * H + unit] : 0.f;
        // loop-invariant shared-memory offsets: this thread's 8 elements of the h operand tile (inside its 64-unit chunk) and
        // the 16-byte chunk it forwards to the peer
        uint32_t h_off[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) h_off[i] = (uint32_t)(unit >> 6) * H_CHUNK + tc::sw128_offset(col0 + i, unit & 63);
        const int gu = (int)c * UNITS + q * 32 + (lane >> 3) * 8;
        const uint32_t fwd_off = (uint32_t)(gu >> 6) * H_CHUNK + tc::sw128_offset(col0 + (lane & 7), gu & 63);
        bool ok = true;
        for (int s = 0; s < T; ++s) {
            const int t = d == 0 ? s : T - 1 - s;
            const size_t blk = blk_index(d, tile, t, (int)c, ntiles, T, CS);
            // this step's gi: from the prefetch ring, or (FX) bias now + W_i x from the accumulators below
            float gr[8], gz[8], gn[8];
            if (FX) {
#pragma unroll
                for (int i = 0; i < 8; ++i) { gr[i] = bx_r; gz[i] = bx_z; }
            } else {
                const int st = s % NSF;
                if (tid == 0) SCAN_TS(5);
                if (ok) ok = tc::mbar_wait(&in_full[st], (s / NSF) & 1, p.dbg, 0x200 + (s & 0xff));
                const uint4* gp = reinterpret_cast<const uint4*>(sIn + (size_t)st * GI_BLOCK) + tid;
                const uint4 u0 = gp[0], u1 = gp[256], u2 = gp[512];
                const __nv_bfloat16* t8 = reinterpret_cast<const __nv_bfloat16*>(&u0);
#pragma unroll
                for (int i = 0; i < 8; ++i) gr[i] = __bfloat162float(t8[i]);
                t8 = reinterpret_cast<const __nv_bfloat16*>(&u1);
#pragma unroll
                for (int i = 0; i < 8; ++i) gz[i] = __bfloat162float(t8[i]);
                t8 = reinterpret_cast<const __nv_bfloat16*>(&u2);
#pragma unroll
                for (int i = 0; i < 8; ++i) gn[i] = __bfloat162float(t8[i]);
            }
            if (!FX) {
#pragma unroll
                for (int i = 0; i < 8; ++i) asm volatile("" ::"f"(gr[i]), "f"(gz[i]), "f"(gn[i]));     // converted before the wait below
            }
            const int buf = s & 1;
            uint8_t* hb = sH + (size_t)buf * KC * H_CHUNK;
            const uint32_t ta = tmem + ((uint32_t)(q * 32) << 16) + col0;
            const uint32_t par = FX ? (uint32_t)(s & 1) : (uint32_t)((s - 1) & 1);
            float r8[8], z8[8], an[8];
            if (FX || s > 0) {
                if (tid == 0) SCAN_TS(6);
                if (ok) ok = tc::mbar_wait(mma_done, par, p.dbg, 0x600 + (s & 0xff));
                if (tid == 0) SCAN_TS(7);
                if (tid == 224) SCAN_TS(12);
                tc::tcgen05_fence_after();
                tmem_ld8(ta, r8); tmem_ld8(ta + NB, z8);
                if (!FX || s > 0) tmem_ld8(ta + 2 * NB, an);
                if (FX) tmem_ld8(ta + 3 * NB, gn);
                tc::tmem_ld_wait();
                if (FX) {
                    // accumulators read: the control thread may start the input projection of the next step
                    tc::tcgen05_fence_before();
                    __syncwarp();
                    if (lane == 0) tc::mbar_arrive(acc_free);
#pragma unroll
                    for (int i = 0; i < 8; ++i) gn[i] += bx_n;
                    if (s == 0) {
#pragma unroll
                        for (int i = 0; i < 8; ++i) an[i] = 0.f;
                    }
                }
                if (tid == 0) SCAN_TS(8);
            } else {
#pragma unroll
                for (int i = 0; i < 8; ++i) { r8[i] = 0.f; z8[i] = 0.f; an[i] = 0.f; }
            }
            if (s == 0 && has_h0) {
                // step 0 with an initial state: the recurrent product W_hh h0 comes from the caller (no MMA at step 0)
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const float* gp = p.gh0 + ((int64_t)d * B + tile * NB + col0 + i) * 3 * H + unit;
                    r8[i] += gp[0]; z8[i] += gp[H]; an[i] += gp[2 * H];
                }
            }
#pragma unroll
            for (int i = 0; i < 8; ++i) { r8[i] = sigmoid_fast(gr[i] + r8[i]); z8[i] = sigmoid_fast(gz[i] + z8[i]); }
            float hn8[8], n8[8];
            __nv_bfloat16 hv[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                hn8[i] = an[i] + bhn;
                n8[i] = tanh_fast(fmaf(r8[i], hn8[i], gn[i]));
                const float h = fmaf(z8[i], hprev[i] - n8[i], n8[i]);
                hprev[i] = h;
                hv[i] = __float2bfloat16(h);
                *reinterpret_cast<__nv_bfloat16*>(hb + h_off[i]) = hv[i];
            }
            // hand h_t to the control thread (this is the step chain): smem writes -> async proxy, one arrival per
            // warp; everything that only feeds HBM is issued afterwards, off the chain
            if (tid == 0) SCAN_TS(9);
            tc::tcgen05_fence_before();
            if (CS > 1 && s + 1 < T) {
                // peer hand-off without the control thread: after the warp's 2-byte writes, lane L re-reads one 16-byte
                // chunk (8 units of lane group L/8, batch column L%8) and stores it asynchronously into the same place of
                // the peer's operand tile; the store completes its bytes on the peer's h_full (async proxy end to end)
                __syncwarp();
                uint8_t* cp = hb + fwd_off;
                const uint4 v = *reinterpret_cast<const uint4*>(cp);
                tc::st_async_v4(tc::mapa_u32(tc::smem_u32(cp), 1u - c), v, tc::mapa_u32(tc::smem_u32(&h_full[buf]), 1u - c));
            }
            tc::fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(epi_done);
            // the ring slot is released only HERE, after this step's results (which consume every value loaded from the slot)
            // have been written: an arrive right behind the loads was seen to overtake them (the loads sat in the LSU queue behind
            // the previous step's global stores), so the producer's next bulk copy replaced the slot before it had been read
            if (!FX && lane == 0) tc::mbar_arrive(&in_empty[s % NSF]);
            if (tid == 0) SCAN_TS(10);
            if (tid == 224) SCAN_TS(13);
            {
                __nv_bfloat16 sr[8], sz[8], sn[8], shn[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    sr[i] = __float2bfloat16(r8[i]); sz[i] = __float2bfloat16(z8[i]);
                    sn[i] = __float2bfloat16(n8[i]); shn[i] = __float2bfloat16(hn8[i]);
                }
                uint4* gs = reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(p.G) + blk * G_BLOCK) + tid;
                gs[0] = *reinterpret_cast<uint4*>(sr); gs[256] = *reinterpret_cast<uint4*>(sz);
                gs[512] = *reinterpret_cast<uint4*>(sn); gs[768] = *reinterpret_cast<uint4*>(shn);
            }
            reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(p.YB) + blk * YB_BLOCK)[tid] = *reinterpret_cast<uint4*>(hv);
            if (s == T - 1 && p.hn_out) {
#pragma unroll
                for (int i = 0; i < 8; ++i) p.hn_out[((int64_t)d * B + tile * NB + col0 + i) * H + unit] = hprev[i];
            }
            if (tid == 0) SCAN_TS(11);
        }
    }
    tc::tcgen05_fence_before();
    __syncthreads();
    if (CS > 1) tc::cluster_sync_all();        // no CTA leaves while a peer may still target its smem
    if (warp == EPI_WARPS) tc::tmem_dealloc(tmem, fwd_tmem_cols(H, FX));
}

static inline cudaError_t launch_fwd(const FwdParams& p_in, cudaStream_t st) {
    FwdParams p = p_in;
    {
        const uint64_t dims[2] = {(uint64_t)p.D * p.H, (uint64_t)p.T * p.B};
        const uint64_t strides[1] = {(uint64_t)p.D * p.H * 2};
        const uint32_t box[2] = {64u, (uint32_t)NB};
        if (make_tmap_bf16(&p.tmY, p.Yrow, 2, dims, strides, box) != 0) return cudaErrorInvalidValue;
    }
    const int CS = p.H / UNITS;
    if (p.H != 128 && p.H != 256) return cudaErrorInvalidValue;
    const bool fx = p.fuse_x != 0;
    if (fx) {
        const uint64_t dx[2] = {64u, p.x_win ? (uint64_t)(p.T + p.B - 1) : (uint64_t)p.T * p.B};
        const uint64_t sx[1] = {64u * 2};
        const uint32_t bx[2] = {64u, (uint32_t)NB};
        const uint64_t dw[2] = {64u, (uint64_t)p.D * 3 * p.H};
        const uint32_t bw[2] = {64u, (uint32_t)UNITS};
        if (make_tmap_bf16(&p.tmX, p.Xrow, 2, dx, sx, bx) != 0 || make_tmap_bf16(&p.tmW, p.Wih, 2, dw, sx, bw) != 0) return cudaErrorInvalidValue;
    }
    const size_t smem = fwd_smem_bytes(p.H, fx);
    void (*kern)(FwdParams) = p.H == 128 ? (fx ? gru_scan_fwd_kernel<128, true> : gru_scan_fwd_kernel<128, false>)
                                         : (fx ? gru_scan_fwd_kernel<256, true> : gru_scan_fwd_kernel<256, false>);
    {   // the shared-memory opt-in is per device (and cheap): set it on every launch rather than caching it process-wide
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)(p.D * (p.B / NB) * CS));
    cfg.blockDim = dim3(THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = CS; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, p);
}

// ---- packed weights: W_hh fp32 [3H][H] (rows r|z|n) -> Wpk[unit u][g][k] bf16 (row of unit u = its three gate rows)
__global__ void pack_whh_image_kernel(const float* __restrict__ w_hh, __nv_bfloat16* __restrict__ img, int H) {
    const int64_t total = (int64_t)3 * H * H;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int k = i % H;
        const int row = i / H;                 // g*H + unit
        const int g = row / H, unit = row % H;
        img[((int64_t)unit * 3 + g) * H + k] = __float2bfloat16(w_hh[i]);
    }
}

// =================================================================================================
// Backward scan (BPTT).  Same cluster / tiling; the TMEM-resident operand is W_hh^T (A[unit k][q] = W_hh[q][k],
// 128 rows x 3H) and the per-step product is
//     D'[k, b] = sum_q W_hh[q, k] * dgh_{s-1}[b, q]                    (tcgen05.mma M=128 N=16, K = 3H)
// i.e. the recurrent part of dh.  The epilogue thread of hidden unit k adds dY_t and the z-carry, forms the
// gate derivatives from the stash, writes its three dgh values (bf16) into the [16 x 3H] operand tile of
// the next step (locally + DSMEM bulk copy to the peers) and streams out dgi / dgh row-major for the
// weight-gradient GEMMs; bias gradients accumulate in registers over all steps.
// The [16 x 3H] operand tile is double-buffered (2 x 24 KB); the control thread publishes it exactly as in the
// forward kernel.
// Per-step inputs (stash G, blocked h_{t-1} YB, blocked fp32 dY) come through a 3-stage bulk-copy ring.
//   dgi_row bf16 [R][D*3H], dghn_row bf16 [R][D*H]: row-major, consumed as MN-major GEMM operands   (written)
// =================================================================================================
static inline size_t bwd_smem_bytes(int H) {
    const int KC3 = 3 * H / 64;
    return (size_t)2 * KC3 * H_CHUNK + (size_t)2 * (UNITS / 64) * H_CHUNK + (size_t)NSB * BWD_STAGE + (size_t)HEAD_CONST + 1024 + 256;
}
constexpr uint32_t BWD_A_COL = 32;        // accumulator in columns [0, 16), W_hh^T from column 32
__host__ __device__ static inline uint32_t bwd_tmem_cols(int H) { return 32 + 3 * H / 2 <= 256 ? 256u : 512u; }

struct BwdParams {
    int B, T, H, D;
    const __nv_bfloat16* WTimg;     // [D][H units][3H]  rows of W_hh^T, copied to TMEM
    const __nv_bfloat16* G;
    const __nv_bfloat16* YB;        // blocked h (see forward)
    const float* dYB;               // blocked fp32 dY: [block][256][8]   (lower layers)
    const float* h0;                // nullable [D][B][H]: h_prev of the first forward step
    float* dh0;                     // nullable [D][B][H]: gradient of the initial hidden state
    // top layer: dY is formed on the fly from the head (biGRU_model.py:111-137): d(concat) = dlogits x lin_w,
    // dY_t[b,u] = davg/T + (argmax_t == t ? dmax : 0), initial carry = d(last hidden); dYB is not read then
    const float* dlogits;           // [B][C] nullable (non-null selects top-layer mode)
    const float* lin_w;             // [C][3H]
    const int* arg;                 // [B][H] argmax_t of the pooled output
    int C;
    __nv_bfloat16* dgi_row;         // [R][D*3H]  (da_r, da_z, da_n)      written by TMA tile stores (tmGI)
    __nv_bfloat16* dghn_row;        // [R][D*H]   da_n * r  (the n-gate column block of dgh)   (tmGN)
    CUtensorMap tmGI, tmGN;         // box 64 x 16, 128B swizzle (filled by launch_bwd)
    float* db_ih;                   // grads of b_ih for direction 0; direction d at + d*dir_stride
    float* db_hh;
    int64_t dir_stride;
    unsigned int* dbg;
#ifdef BIGRU_SCAN_TIMING
    unsigned long long* ts;
#endif
};

// K chunks [u0, u0 + NCH) of each of the three gate blocks of the [16 x 3H] dgh tile, fully unrolled (see fwd_issue_group)
template <int H, int NCH, bool FIRST>
__device__ __forceinline__ void bwd_issue_group(uint32_t tmem_d, uint32_t tmem_a_grp, uint64_t desc_grp) {
    constexpr uint32_t idesc = tc::umma_idesc_bf16(UNITS, NB);
    constexpr int KC = H / 64;
#pragma unroll
    for (int g = 0; g < 3; ++g) {
#pragma unroll
        for (int u = 0; u < NCH; ++u) {
#pragma unroll
            for (int kk = 0; kk < 4; ++kk)
                umma_bf16_ts(tmem_d, tmem_a_grp + (uint32_t)(((g * KC + u) * 4 + kk) * 8),
                             desc_grp + (uint64_t)((g * KC + u) * (H_CHUNK >> 4) + 2 * kk), idesc, (FIRST && g == 0 && u == 0 && kk == 0) ? 0u : 1u);
        }
    }
}

template <int H>
__global__ void __launch_bounds__(THREADS, 1) gru_scan_bwd_kernel(const __grid_constant__ BwdParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    constexpr int KC = H / 64, KC3 = 3 * KC, CS = H / UNITS, MYCH = UNITS / 64;
    const int B = p.B, T = p.T, D = p.D;
    uint8_t* sD = smem;                                    // [2][KC3][H_CHUNK]  dgh operand tiles
    uint8_t* sN = sD + (size_t)2 * KC3 * H_CHUNK;          // [2][UNITS/64][H_CHUNK]  da_n of this CTA's units (dgi n-gate, store only)
    uint8_t* sIn = sN + (size_t)2 * (UNITS / 64) * H_CHUNK;   // [NSB][G | YB | dY]
    float* sHead = reinterpret_cast<float*>(sIn + (size_t)NSB * BWD_STAGE);    // [3][256][8]
    uint64_t* bars = reinterpret_cast<uint64_t*>(sIn + (size_t)NSB * BWD_STAGE + HEAD_CONST);
    uint64_t* d_full = bars;           // [2]  peers' dgh chunks landed
    uint64_t* mma_done = bars + 2;
    uint64_t* epi_done = bars + 3;
    uint64_t* in_full = bars + 4;      // [NSB]
    uint64_t* in_empty = bars + 4 + NSB;   // [NSB]
    uint64_t* st_done = bars + 4 + 2 * NSB;    // n-gate tile written (only the TMA row stores wait for it)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 5 + 2 * NSB);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t c = CS > 1 ? tc::cluster_ctarank() : 0u;
    const int cluster_id = blockIdx.x / CS;
    const int ntiles = B / NB;
    const int d = cluster_id / ntiles, tile = cluster_id % ntiles;
    const int64_t R = (int64_t)T * B;
    const bool top = p.dlogits != nullptr;

    if (threadIdx.x == 0) {
        tc::mbar_init(&d_full[0], 1);
        tc::mbar_init(&d_full[1], 1);
        tc::mbar_init(mma_done, 1);
        tc::mbar_init(epi_done, EPI_WARPS);
        tc::mbar_init(st_done, EPI_WARPS);
        for (int i = 0; i < NSB; ++i) { tc::mbar_init(&in_full[i], 1); tc::mbar_init(&in_empty[i], EPI_WARPS); }
        tc::fence_mbar_init();
    }
    if (warp == EPI_WARPS) tc::tmem_alloc(tmem_slot, bwd_tmem_cols(H));
    tc::tcgen05_fence_before();
    __syncthreads();
    if (CS > 1) tc::cluster_sync_all();
    tc::tcgen05_fence_after();
    const uint32_t tmem = *tmem_slot;
    const uint32_t gate_bytes_mine = (uint32_t)(UNITS / 64) * H_CHUNK;     // per gate: 2 chunks = 4 KB
    if (warp < EPI_WARPS)
        load_weights_to_tmem(p.WTimg + ((size_t)d * CS + c) * UNITS * 3 * H, 3 * H, tmem, BWD_A_COL, warp, lane);
    tc::tcgen05_fence_before();
    __syncthreads();
    tc::tcgen05_fence_after();

    if (warp == EPI_WARPS + 1) {
        // ---- input prefetch ring: stash + blocked h_{t-1} + blocked dY of each step, up to NSB steps ahead
        if (tc::elect_one()) {
            bool ok = true;
            for (int s = 0; s < T; ++s) {
                const int st = s % NSB;
                if (s >= NSB && ok) ok = tc::mbar_wait(&in_empty[st], ((s / NSB) - 1) & 1, p.dbg, 0x300 + (s & 0xff));
                const int t = d == 0 ? T - 1 - s : s;
                const bool first = d == 0 ? t == 0 : t == T - 1;         // first step of the FORWARD recurrence: h_prev = 0
                uint8_t* dst = sIn + (size_t)st * BWD_STAGE;
                tc::mbar_arrive_expect_tx(&in_full[st], (uint32_t)(G_BLOCK + (top ? 0 : DY_BLOCK) + (first ? 0 : YB_BLOCK)));
                const size_t blk = blk_index(d, tile, t, (int)c, ntiles, T, CS);
                tc::bulk_g2s(dst, reinterpret_cast<const uint8_t*>(p.G) + blk * G_BLOCK, G_BLOCK, &in_full[st]);
                if (!top) tc::bulk_g2s(dst + G_BLOCK + YB_BLOCK, reinterpret_cast<const uint8_t*>(p.dYB) + blk * DY_BLOCK, DY_BLOCK, &in_full[st]);
                if (!first) {
                    const size_t pblk = blk_index(d, tile, d == 0 ? t - 1 : t + 1, (int)c, ntiles, T, CS);
                    tc::bulk_g2s(dst + G_BLOCK, reinterpret_cast<const uint8_t*>(p.YB) + pblk * YB_BLOCK, YB_BLOCK, &in_full[st]);
                }
            }
        }
    } else if (warp == EPI_WARPS) {
        // ---- control thread (see forward kernel)
        if (tc::elect_one()) {
            bool ok = true;
            const int Tend = T + (p.dh0 ? 1 : 0);          // one more product (no gate math) when d(h0) is wanted
            if (CS > 1 && Tend > 1) tc::mbar_arrive_expect_tx(&d_full[0], (uint32_t)(CS - 1) * 3 * gate_bytes_mine);
            auto store_tile = [&](int step) {             // dgi / dgh_n rows of time step `step`, this CTA's 128 units
                const int tt = d == 0 ? T - 1 - step : step;
                const int row = tt * B + tile * NB;
                const uint8_t* tb = sD + (size_t)(step & 1) * KC3 * H_CHUNK;
                const uint8_t* nb = sN + (size_t)(step & 1) * MYCH * H_CHUNK;
                for (int k = 0; k < MYCH; ++k) {
                    const int cu = (int)c * UNITS + 64 * k;
                    const size_t co = ((size_t)c * MYCH + k) * H_CHUNK;
                    tc::tma_store_2d(&p.tmGI, tb + (size_t)(0 * KC) * H_CHUNK + co, d * 3 * H + cu, row);            // da_r
                    tc::tma_store_2d(&p.tmGI, tb + (size_t)(1 * KC) * H_CHUNK + co, d * 3 * H + H + cu, row);        // da_z
                    tc::tma_store_2d(&p.tmGI, nb + (size_t)k * H_CHUNK, d * 3 * H + 2 * H + cu, row);                 // da_n
                    tc::tma_store_2d(&p.tmGN, tb + (size_t)(2 * KC) * H_CHUNK + co, d * H + cu, row);                // da_n * r
                }
                tc::tma_store_commit();
            };
            // operand bases: inside each gate block, K chunks [2c, 2c+2) are this CTA's own (local group)
            const uint32_t a_loc = tmem + BWD_A_COL + (uint32_t)c * (MYCH * 32);
            const uint32_t a_rem = tmem + BWD_A_COL + (uint32_t)(1 - (int)c) * (MYCH * 32);
            const uint32_t db0 = tc::smem_u32(sD);
            const uint64_t d_loc0 = tc::umma_desc_k_sw128(db0 + (uint32_t)c * gate_bytes_mine);
            const uint64_t d_rem0 = tc::umma_desc_k_sw128(db0 + (uint32_t)(1 - (int)c) * gate_bytes_mine);
            constexpr uint64_t BUF_DESC = (uint64_t)((KC3 * H_CHUNK) >> 4);
            for (int s = 1; s < Tend; ++s) {
                const int pb = (s - 1) & 1;
                if (ok) ok = tc::mbar_wait(epi_done, (s - 1) & 1, p.dbg, 0x700 + (s & 0xff));
                SCAN_TS(0);
                tc::tcgen05_fence_after();
                if (CS > 1) {
                    bwd_issue_group<H, MYCH, true>(tmem, a_loc, d_loc0 + (pb ? BUF_DESC : 0));
                    SCAN_TS(1);
                    if (ok) ok = tc::mbar_wait(&d_full[pb], ((s - 1) >> 1) & 1, p.dbg, 0x800 + (s & 0xff));
                    SCAN_TS(2);
                    if (s + 1 < Tend) tc::mbar_arrive_expect_tx(&d_full[s & 1], (uint32_t)(CS - 1) * 3 * gate_bytes_mine);
                    tc::tcgen05_fence_after();
                    bwd_issue_group<H, MYCH, false>(tmem, a_rem, d_rem0 + (pb ? BUF_DESC : 0));
                } else {
                    bwd_issue_group<H, KC, true>(tmem, a_loc, d_loc0 + (pb ? BUF_DESC : 0));
                }
                tc::tma_store_wait_read();
                tc::umma_commit(mma_done);
                SCAN_TS(3);
                if (ok) ok = tc::mbar_wait(st_done, (s - 1) & 1, p.dbg, 0xa00 + (s & 0xff));
                store_tile(s - 1);
            }
            if (Tend == T) {
                if (ok) ok = tc::mbar_wait(epi_done, (T - 1) & 1, p.dbg, 0x700);
                if (ok) ok = tc::mbar_wait(st_done, (T - 1) & 1, p.dbg, 0xa00);
                store_tile(T - 1);
            }
            tc::tma_store_wait_all();
        }
    } else if (warp < EPI_WARPS) {
        const int q = warp & 3, half = warp >> 2;
        const int j = q * 32 + lane;
        const int unit = (int)c * UNITS + j;
        const int col0 = half * 8;
        const int tid = threadIdx.x;
        float dhz[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) dhz[i] = 0.f;
        // top layer: d(concat) rows of this thread's 8 batch columns ([last | max | avg] x lin_w^T) stay in registers for all steps
        float h_avg[8], h_max[8];
        int h_arg[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) { h_avg[i] = 0.f; h_max[i] = 0.f; h_arg[i] = -1; }
        if (top) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int b = tile * NB + col0 + i;
                float dl = 0.f, dm = 0.f, da = 0.f;
                for (int cc = 0; cc < p.C; ++cc) {
                    const float g = p.dlogits[(int64_t)b * p.C + cc];
                    const float* w = p.lin_w + (int64_t)cc * 3 * H;
                    dl = fmaf(g, w[unit], dl); dm = fmaf(g, w[H + unit], dm); da = fmaf(g, w[2 * H + unit], da);
                }
                dhz[i] = dl;                                   // d(last hidden) enters the carry of both directions
                h_avg[i] = da / (float)T; h_max[i] = dm; h_arg[i] = p.arg[(int64_t)b * H + unit];
            }
        }
        float sb_r = 0.f, sb_z = 0.f, sb_n = 0.f, sb_nr = 0.f;
        // loop-invariant shared-memory offsets (see forward kernel)
        uint32_t e_off[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) e_off[i] = tc::sw128_offset(col0 + i, unit & 63);
        const int kc_u = unit >> 6;
        const int gu = (int)c * UNITS + q * 32 + (lane >> 3) * 8;
        const uint32_t fwd_off = (uint32_t)(gu >> 6) * H_CHUNK + tc::sw128_offset(col0 + (lane & 7), gu & 63);
        const int Tend = T + (p.dh0 ? 1 : 0);              // the dgh of the last step also feeds d(h0) (control thread)
        bool ok = true;
        for (int s = 0; s < T; ++s) {
            const int t = d == 0 ? T - 1 - s : s;
            const bool first = d == 0 ? t == 0 : t == T - 1;
            const int64_t row0 = (int64_t)t * B + tile * NB + col0;
            float vr[8], vz[8], vn[8], vhn[8], vhp[8], vdy[8];
            {
                const int st = s % NSB;
                if (tid == 0) SCAN_TS(5);
                if (ok) ok = tc::mbar_wait(&in_full[st], (s / NSB) & 1, p.dbg, 0x200 + (s & 0xff));
                if (tid == 0) SCAN_TS(6);
                const uint8_t* base = sIn + (size_t)st * BWD_STAGE;
                const uint4* gp = reinterpret_cast<const uint4*>(base) + tid;
                const uint4 u0 = gp[0], u1 = gp[256], u2 = gp[512], u3 = gp[768];
                const uint4 uh = first ? make_uint4(0u, 0u, 0u, 0u) : reinterpret_cast<const uint4*>(base + G_BLOCK)[tid];
                float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
                if (!top) {
                    const float4* dyp = reinterpret_cast<const float4*>(base + G_BLOCK + YB_BLOCK) + 2 * tid;
                    a = dyp[0]; b = dyp[1];
                }
                const __nv_bfloat16* t8 = reinterpret_cast<const __nv_bfloat16*>(&u0);
#pragma unroll
                for (int i = 0; i < 8; ++i) vr[i] = __bfloat162float(t8[i]);
                t8 = reinterpret_cast<const __nv_bfloat16*>(&u1);
#pragma unroll
                for (int i = 0; i < 8; ++i) vz[i] = __bfloat162float(t8[i]);
                t8 = reinterpret_cast<const __nv_bfloat16*>(&u2);
#pragma unroll
                for (int i = 0; i < 8; ++i) vn[i] = __bfloat162float(t8[i]);
                t8 = reinterpret_cast<const __nv_bfloat16*>(&u3);
#pragma unroll
                for (int i = 0; i < 8; ++i) vhn[i] = __bfloat162float(t8[i]);
                t8 = reinterpret_cast<const __nv_bfloat16*>(&uh);
#pragma unroll
                for (int i = 0; i < 8; ++i) vhp[i] = __bfloat162float(t8[i]);
                if (first && p.h0) {                        // the caller's initial state, in fp32
#pragma unroll
                    for (int i = 0; i < 8; ++i) vhp[i] = p.h0[((int64_t)d * B + tile * NB + col0 + i) * H + unit];
                }
                vdy[0] = a.x; vdy[1] = a.y; vdy[2] = a.z; vdy[3] = a.w; vdy[4] = b.x; vdy[5] = b.y; vdy[6] = b.z; vdy[7] = b.w;
                if (top) {                                  // dY_t = davg / T + (argmax_t == t ? dmax : 0)
#pragma unroll
                    for (int i = 0; i < 8; ++i) vdy[i] = h_avg[i] + (h_arg[i] == t ? h_max[i] : 0.f);
                }
            }
            // everything that does not depend on the recurrent product is formed before the wait on the tensor pipe
            float c_n[8], c_r[8], c_z[8], pre[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float r = vr[i], z = vz[i], n = vn[i];
                c_n[i] = (1.f - z) * (1.f - n * n);                 // da_n = dh * c_n
                c_r[i] = vhn[i] * r * (1.f - r);                    // da_r = da_n * c_r
                c_z[i] = (vhp[i] - n) * z * (1.f - z);              // da_z = dh * c_z
                pre[i] = dhz[i] + vdy[i];
            }
            // pin these values BEFORE the spin on the tensor pipe (the compiler otherwise sinks the arithmetic below the wait,
            // onto the step chain)
#pragma unroll
            for (int i = 0; i < 8; ++i) asm volatile("" ::"f"(c_n[i]), "f"(c_r[i]), "f"(c_z[i]), "f"(pre[i]), "f"(vr[i]), "f"(vz[i]));
            float acc[8];
            if (s > 0) {
                if (tid == 0) SCAN_TS(4);
                if (ok) ok = tc::mbar_wait(mma_done, (s - 1) & 1, p.dbg, 0x900 + (s & 0xff));
                if (tid == 0) SCAN_TS(7);
                tc::tcgen05_fence_after();
                tmem_ld8(tmem + ((uint32_t)(q * 32) << 16) + col0, acc);
                tc::tmem_ld_wait();
                if (tid == 0) SCAN_TS(8);
            } else {
#pragma unroll
                for (int i = 0; i < 8; ++i) acc[i] = 0.f;
            }
            const int buf = s & 1;
            uint8_t* tileb = sD + (size_t)buf * KC3 * H_CHUNK;
            uint8_t* t_r = tileb + (size_t)(0 * KC + kc_u) * H_CHUNK;
            uint8_t* t_z = tileb + (size_t)(1 * KC + kc_u) * H_CHUNK;
            uint8_t* t_n = tileb + (size_t)(2 * KC + kc_u) * H_CHUNK;
            float dar[8], daz[8], dan[8], danr[8];
            __nv_bfloat16 dan_bf[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float dh = acc[i] + pre[i];
                dan[i] = dh * c_n[i];
                dar[i] = dan[i] * c_r[i];
                daz[i] = dh * c_z[i];
                danr[i] = dan[i] * vr[i];
                dhz[i] = dh * vz[i];
                // one packed conversion per two values (the conversion pipe is the narrow one here)
                const __nv_bfloat162 rz = __floats2bfloat162_rn(dar[i], daz[i]);
                *reinterpret_cast<__nv_bfloat16*>(t_r + e_off[i]) = rz.x;
                *reinterpret_cast<__nv_bfloat16*>(t_z + e_off[i]) = rz.y;
                const __nv_bfloat162 nn = __floats2bfloat162_rn(danr[i], dan[i]);
                *reinterpret_cast<__nv_bfloat16*>(t_n + e_off[i]) = nn.x;
                dan_bf[i] = nn.y;
            }
            // hand dgh_s to the tensor pipe (the step chain): own chunks -> peer with st.async (see forward kernel), then
            // the local arrival; the n-gate tile (TMA store only) and the bias sums follow, off the chain
            if (tid == 0) SCAN_TS(9);
            tc::tcgen05_fence_before();
            if (CS > 1 && s + 1 < Tend) {
                __syncwarp();
                const uint32_t rbar = tc::mapa_u32(tc::smem_u32(&d_full[buf]), 1u - c);
#pragma unroll
                for (int g = 0; g < 3; ++g) {
                    uint8_t* cp = tileb + (size_t)(g * KC) * H_CHUNK + fwd_off;
                    const uint4 v = *reinterpret_cast<const uint4*>(cp);
                    tc::st_async_v4(tc::mapa_u32(tc::smem_u32(cp), 1u - c), v, rbar);
                }
            }
            tc::fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(epi_done);
            // the ring slot is released only HERE, after this step's results (which consume every value loaded from the slot)
            // have been written: an arrive right behind the loads was seen to overtake them (the loads sat in the LSU queue behind
            // the previous step's global stores), so the producer's next bulk copy replaced the slot before it had been read
            if (lane == 0) tc::mbar_arrive(&in_empty[s % NSB]);
            if (tid == 0) SCAN_TS(10);
#pragma unroll
            for (int i = 0; i < 8; ++i)
                *reinterpret_cast<__nv_bfloat16*>(sN + (size_t)(buf * MYCH + ((unit & (UNITS - 1)) >> 6)) * H_CHUNK + e_off[i]) = dan_bf[i];
            tc::fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(st_done);
#pragma unroll
            for (int i = 0; i < 8; ++i) { sb_r += dar[i]; sb_z += daz[i]; sb_n += dan[i]; sb_nr += danr[i]; }
            if (tid == 0) SCAN_TS(11);
        }
        // bias gradients: sum the 8 columns of this thread; the two column halves and all tiles add atomically
        float* dbi = p.db_ih + (int64_t)d * p.dir_stride;
        float* dbh = p.db_hh + (int64_t)d * p.dir_stride;
        atomicAdd(dbi + unit, sb_r); atomicAdd(dbi + H + unit, sb_z); atomicAdd(dbi + 2 * H + unit, sb_n);
        atomicAdd(dbh + unit, sb_r); atomicAdd(dbh + H + unit, sb_z); atomicAdd(dbh + 2 * H + unit, sb_nr);
        if (p.dh0) {
            // gradient of the initial hidden state = z-carry of the last step + W_hh^T dgh of the last step (one more product)
            float acc[8];
            if (ok) ok = tc::mbar_wait(mma_done, (T - 1) & 1, p.dbg, 0x900);
            tc::tcgen05_fence_after();
            tmem_ld8(tmem + ((uint32_t)(q * 32) << 16) + col0, acc);
            tc::tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 8; ++i) p.dh0[((int64_t)d * B + tile * NB + col0 + i) * H + unit] = dhz[i] + acc[i];
        }
    }
    tc::tcgen05_fence_before();
    __syncthreads();
    if (CS > 1) tc::cluster_sync_all();
    if (warp == EPI_WARPS) tc::tmem_dealloc(tmem, bwd_tmem_cols(H));
}

static inline cudaError_t launch_bwd(const BwdParams& p_in, cudaStream_t st) {
    BwdParams p = p_in;
    {
        const uint32_t box[2] = {64u, (uint32_t)NB};
        const uint64_t d1[2] = {(uint64_t)p.D * 3 * p.H, (uint64_t)p.T * p.B};
        const uint64_t s1[1] = {(uint64_t)p.D * 3 * p.H * 2};
        const uint64_t d2[2] = {(uint64_t)p.D * p.H, (uint64_t)p.T * p.B};
        const uint64_t s2[1] = {(uint64_t)p.D * p.H * 2};
        if (make_tmap_bf16(&p.tmGI, p.dgi_row, 2, d1, s1, box) != 0 || make_tmap_bf16(&p.tmGN, p.dghn_row, 2, d2, s2, box) != 0)
            return cudaErrorInvalidValue;
    }
    const int CS = p.H / UNITS;
    if (p.H != 128 && p.H != 256) return cudaErrorInvalidValue;
    const size_t smem = bwd_smem_bytes(p.H);
    void (*kern)(BwdParams) = p.H == 128 ? gru_scan_bwd_kernel<128> : gru_scan_bwd_kernel<256>;
    {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)(p.D * (p.B / NB) * CS));
    cfg.blockDim = dim3(THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = CS; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, p);
}

// W_hh fp32 [3H][H] -> packed W_hh^T: WTpk[unit k][q] = W_hh[q][k]   (row of unit k = column k of W_hh, 3H long)
__global__ void pack_whhT_image_kernel(const float* __restrict__ w_hh, __nv_bfloat16* __restrict__ img, int H) {
    const int64_t total = (int64_t)3 * H * H;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int k = i % H;                   // hidden unit (column of W_hh)
        const int qrow = i / H;                // gate row q
        img[(int64_t)k * 3 * H + qrow] = __float2bfloat16(w_hh[i]);
    }
}

}  // namespace tcs
