// tc_scan_w.cuh - persistent GRU recurrence on tcgen05 tensor cores for WIDE hidden sizes (H = 512: BASELINE.json configs[4],
// /root/reference/biGRU_model.py:32-33 accepts any hidden_size), bf16 operands, fp32 accumulate / state.
//
// Tensor memory (512 columns x 128 lanes x 32 bit per SM) cannot hold a 128-unit slice of W_hh at H = 512 (3 x 128 x 512 bf16 =
// 768 columns).  So a thread-block CLUSTER of CS = H/64 = 8 CTAs walks all T steps of one (direction, 32-row batch tile); CTA c
// owns hidden units [64c, 64c+64).  Geometry, blocked layouts and the exchange protocols are those of tc_scan_x.cuh (the
// fp32-class kernels) with single bf16 operands.
//
// Forward (output-partitioned, all-gather of h).  The A operand rows are STACKED BY GATE: TMEM lanes 0-63 = W_hr rows of the
// CTA's units, lanes 64-127 = W_hz rows (256 columns for K = 512); the W_hn rows sit on lanes 0-63 of a second column group.
// 64 (accumulators) + 256 + 256 columns do not fit, so the n-gate weights of the LAST two K chunks (128 of 512 columns of
// W_hn) stay in shared memory and enter as SS-mode MMAs (8 of the 64 MMAs of a step):
//     D_rz[lane, b] = sum_k A_rz[lane, k] h[b, k]      D_n[unit, b] = sum_k W_hn[unit, k] h[b, k]
// r and n of a unit come out on lane `unit`, z on lane 64 + unit: the warps of lanes 64-127 and 0-63 swap half of their
// columns through shared memory, after which every thread owns one unit x 8 batch columns (as in tc_scan_x.cuh).
//
// Backward (reduction-partitioned, reduce-scatter of dh): CTA c keeps the W_hh rows of ITS OWN units' gates (K index
// kq = g*64 + jj, 192 wide) for ALL H output units k as H/128 row blocks of 128 lanes, multiplies them with its local dgh tile
// [32 x 192] and sends the fp32 partial sums of units it does not own to their owners (st.async into a receive buffer).
//
// Blocked layouts (time-major): block (d, tile, t, cta) = (((d*ntiles + tile)*T + t)*CS + cta), inside a block
// [gate][thread 0..255][8 batch columns], thread tid = j + 64*(cb/8) <-> unit j = tid % 64 of the CTA, columns [8*(tid/64), +8):
//   giW  bf16 [block][3][256][8]   input projection incl. b_ih (+ b_hh for r, z)   (tc_gemm OUT_SCAN_BF16, U = 64, NB = 32)  read
//   GW   bf16 [block][4][256][8]   r, z, n, W_hn h + b_hn                           stash, written fwd / read bwd
//   YBW  bf16 [block][256][8]      h_t                                              written fwd / read bwd
//   dYBW fp32 [block][256][8]      dL/dy_t (lower layers)                           (tc_gemm OUT_SCAN_F32)  read
//   Yrow bf16 [R][D*H], dgi_row bf16 [R][D*3H], dghn_row bf16 [R][D*H]             row-major GEMM operands
#pragma once
#include "tc_common.cuh"
#include "tc_scan.cuh"
#include "tc_scan_x.cuh"

namespace tcw {

using tcx::NB;            // 32 batch rows per tile
using tcx::UNITS;         // 64 hidden units per CTA
using tcx::EPI_WARPS;
using tcx::THREADS;
using tcx::H_CHUNK;       // [32 x 64] bf16 K-major chunk, 128B swizzle: 4 KB
using tcx::blk_index;
using tcx::tmem_ld16f;
using tcx::tmem_ld_wait_pin;
using tcx::epi_barrier;

constexpr int GI_BLOCK = 3 * 256 * 16;
constexpr int G_BLOCK = 4 * 256 * 16;
constexpr int YB_BLOCK = 256 * 16;
constexpr int DY_BLOCK = 256 * 32;
constexpr int NSF = 4, NSB = 2;
constexpr int XBUF_BYTES = 8 * 4 * 32 * 16;        // forward lane-half exchange: [warp][slot 0..3][lane] float4
constexpr int BWD_STAGE = G_BLOCK + YB_BLOCK + DY_BLOCK;
constexpr uint32_t D_RZ = 0, D_N = 32, A_RZ = 64;  // forward TMEM columns: accumulators, then the stacked r|z weights
constexpr int TAIL_TILE = 128 * 128;               // one [128 rows x 64 k] bf16 K-major tile of the n-gate tail (rows 64.. are zero)

template <int H>
struct Geo {
    static constexpr int KC = H / 64, CS = H / 64;
    static constexpr uint32_t A_N = A_RZ + H / 2;                                   // n-gate weight columns
    static constexpr int KC_T = ((512 - (int)A_N) / 32) < KC ? ((512 - (int)A_N) / 32) : KC;   // n-gate K chunks resident in TMEM
    static constexpr int NTAIL = KC - KC_T;                                         // ... and in shared memory
    static constexpr int ROW_ELEMS = H + KC_T * 64;                                 // bf16 per lane of the forward TMEM image
    static constexpr int NRB = H / 128;                                             // backward row blocks
    static constexpr int RECV_BYTES = CS * 8 * 64 * 16;                             // [src cta][column group][unit j] float4
};

static inline size_t fwd_smem_bytes(int H) {
    const int KC = H / 64;
    const int ntail = H == 512 ? 2 : 0;
    return (size_t)2 * KC * H_CHUNK + (size_t)ntail * TAIL_TILE + (size_t)NSF * GI_BLOCK + XBUF_BYTES + 1024 + 512;
}
static inline size_t bwd_smem_bytes(int H) {
    const int CS = H / 64;
    return (size_t)2 * 3 * H_CHUNK + (size_t)2 * H_CHUNK + (size_t)2 * CS * 8 * 64 * 16 + (size_t)NSB * BWD_STAGE + 1024 + 512;
}

struct FwdParams {
    int B, T, H, D;
    const __nv_bfloat16* Wimg;    // [D][CS][128 lanes][ROW_ELEMS]  then  [D][CS][NTAIL][128 rows][64] (see pack_wide_images_kernel)
    const __nv_bfloat16* Wtail;
    const __nv_bfloat16* giW;
    const float* b_hn;            // [D][H]
    __nv_bfloat16* GW;
    __nv_bfloat16* YBW;
    float* hn_out;                // nullable [D][B][H]
    const float* h0;              // nullable [D][B][H]: initial hidden state of this layer ...
    const float* gh0;             // ... and its recurrent product W_hh h0 [D][B][3H] (fp32, no bias, formed by the caller): step 0 reads it
    __nv_bfloat16* Yrow;          // [R][D*H]
    unsigned int* dbg;
    CUtensorMap tmY;              // box 64 x 32 (filled by launch_fwd)
};

// K chunk u of h against the stacked r|z rows and the n rows (TMEM-resident part): 8 MMAs
template <bool FIRST>
__device__ __forceinline__ void fwd_issue_chunk_ts(uint32_t tmem, uint32_t a_rz, uint32_t a_n, uint64_t desc_b) {
    constexpr uint32_t idesc = tc::umma_idesc_bf16(128, NB);
#pragma unroll
    for (int kk = 0; kk < 4; ++kk)
        tcs::umma_bf16_ts(tmem + D_RZ, a_rz + (uint32_t)(kk * 8), desc_b + (uint64_t)(2 * kk), idesc, (FIRST && kk == 0) ? 0u : 1u);
#pragma unroll
    for (int kk = 0; kk < 4; ++kk)
        tcs::umma_bf16_ts(tmem + D_N, a_n + (uint32_t)(kk * 8), desc_b + (uint64_t)(2 * kk), idesc, (FIRST && kk == 0) ? 0u : 1u);
}
// ... the same with the n rows from shared memory (tail chunks)
template <bool FIRST>
__device__ __forceinline__ void fwd_issue_chunk_ss(uint32_t tmem, uint32_t a_rz, uint64_t desc_wn, uint64_t desc_b) {
    constexpr uint32_t idesc = tc::umma_idesc_bf16(128, NB);
#pragma unroll
    for (int kk = 0; kk < 4; ++kk)
        tcs::umma_bf16_ts(tmem + D_RZ, a_rz + (uint32_t)(kk * 8), desc_b + (uint64_t)(2 * kk), idesc, (FIRST && kk == 0) ? 0u : 1u);
#pragma unroll
    for (int kk = 0; kk < 4; ++kk)
        tc::umma_bf16(tmem + D_N, desc_wn + (uint64_t)(2 * kk), desc_b + (uint64_t)(2 * kk), idesc, (FIRST && kk == 0) ? 0u : 1u);
}

__device__ __forceinline__ void unpack8(const uint4& u, float (&f)[8]) {
    const __nv_bfloat16* t8 = reinterpret_cast<const __nv_bfloat16*>(&u);
#pragma unroll
    for (int i = 0; i < 8; ++i) f[i] = __bfloat162float(t8[i]);
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        __nv_bfloat162 h2 = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
        w[i] = *reinterpret_cast<uint32_t*>(&h2);
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
}

template <int H>
__global__ void __launch_bounds__(THREADS, 1) gru_scanw_fwd_kernel(const __grid_constant__ FwdParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    using G = Geo<H>;
    constexpr int KC = G::KC, CS = G::CS, KC_T = G::KC_T, NTAIL = G::NTAIL;
    constexpr int TILE_BYTES = KC * H_CHUNK;               // one h operand tile [32 x H]
    const int B = p.B, T = p.T;
    uint8_t* sH = smem;                                    // [2 buf][KC][H_CHUNK]
    uint8_t* sWn = sH + (size_t)2 * TILE_BYTES;            // [NTAIL][TAIL_TILE]
    uint8_t* sIn = sWn + (size_t)NTAIL * TAIL_TILE;        // [NSF][GI_BLOCK]
    uint8_t* sX = sIn + (size_t)NSF * GI_BLOCK;            // exchange buffer
    uint64_t* bars = reinterpret_cast<uint64_t*>(sX + XBUF_BYTES);
    uint64_t* h_full = bars;                 // [2 buf][8 src]
    uint64_t* mma_done = bars + 16;
    uint64_t* epi_done = bars + 17;
    uint64_t* in_full = bars + 18;           // [NSF]
    uint64_t* in_empty = bars + 18 + NSF;    // [NSF]
    uint64_t* xch = bars + 18 + 2 * NSF;     // [8]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 26 + 2 * NSF);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t c = tc::cluster_ctarank();
    const int cluster_id = blockIdx.x / CS;
    const int ntiles = B / NB;
    const int d = cluster_id / ntiles, tile = cluster_id % ntiles;

    if (threadIdx.x == 0) {
        for (int i = 0; i < 16; ++i) tc::mbar_init(&h_full[i], 1);
        tc::mbar_init(mma_done, 1);
        tc::mbar_init(epi_done, EPI_WARPS);
        for (int i = 0; i < NSF; ++i) { tc::mbar_init(&in_full[i], 1); tc::mbar_init(&in_empty[i], EPI_WARPS); }
        for (int i = 0; i < EPI_WARPS; ++i) tc::mbar_init(&xch[i], 1);
        // first uses of the per-source "peer chunk landed" barriers (h_s lands in buffer s & 1), armed before the cluster-wide
        // sync so that a fast peer's st.async bytes never reach a barrier that does not expect them
        for (uint32_t u = 0; u < (uint32_t)CS; ++u) {
            if (u == c) continue;
            if (T > 1) tc::mbar_arrive_expect_tx(&h_full[u], H_CHUNK);
            if (T > 2) tc::mbar_arrive_expect_tx(&h_full[8 + u], H_CHUNK);
        }
        tc::fence_mbar_init();
    }
    if (warp == EPI_WARPS) tc::tmem_alloc(tmem_slot, 512);
    // n-gate tail tiles -> shared memory in the UMMA K-major / 128B-swizzle layout (16-byte pieces, piece index ^ row % 8)
    if (NTAIL > 0) {
        const uint4* src = reinterpret_cast<const uint4*>(p.Wtail + ((size_t)d * CS + c) * NTAIL * 128 * 64);
        for (int i = threadIdx.x; i < NTAIL * 128 * 8; i += THREADS) {
            const int tl = i / (128 * 8), row = (i / 8) % 128, c16 = i % 8;
            tc::sts_u4(tc::smem_u32(sWn) + (uint32_t)(tl * TAIL_TILE + row * 128 + ((c16 ^ (row & 7)) << 4)), src[i]);
        }
        tc::fence_proxy_async_smem();
    }
    tc::tcgen05_fence_before();
    __syncthreads();
    tc::cluster_sync_all();
    tc::tcgen05_fence_after();
    const uint32_t tmem = *tmem_slot;
    if (warp < EPI_WARPS)
        tcs::load_weights_to_tmem(p.Wimg + ((size_t)d * CS + c) * 128 * G::ROW_ELEMS, G::ROW_ELEMS, tmem, A_RZ, warp, lane);
    tc::tcgen05_fence_before();
    __syncthreads();
    tc::tcgen05_fence_after();

    if (warp == EPI_WARPS + 1) {
        // ---- input prefetch: one bulk copy (12 KB) per step into the ring
        if (tc::elect_one()) {
            bool ok = true;
            for (int s = 0; s < T; ++s) {
                const int st = s % NSF;
                if (s >= NSF && ok) ok = tc::mbar_wait(&in_empty[st], ((s / NSF) - 1) & 1, p.dbg, 0x3300 + (s & 0xff));
                const int t = d == 0 ? s : T - 1 - s;
                tc::mbar_arrive_expect_tx(&in_full[st], GI_BLOCK);
                tc::bulk_g2s(sIn + (size_t)st * GI_BLOCK,
                             reinterpret_cast<const uint8_t*>(p.giW) + blk_index(d, tile, t, (int)c, ntiles, T, CS) * GI_BLOCK,
                             GI_BLOCK, &in_full[st]);
            }
        }
    } else if (warp == EPI_WARPS) {
        // ---- control thread: 64 MMAs per step; K chunk u is multiplied as soon as source CTA u's bytes have landed
        if (tc::elect_one()) {
            bool ok = true;
            uint32_t epi_rounds = 0, hf_use0 = 0, hf_use1 = 0;
            auto store_tile = [&](int step) {             // this CTA's 64 columns of Yrow for time step `step`
                const int tt = d == 0 ? step : T - 1 - step;
                tc::tma_store_2d(&p.tmY, sH + (size_t)(step & 1) * TILE_BYTES + (size_t)c * H_CHUNK, d * H + (int)c * UNITS, tt * B + tile * NB);
                tc::tma_store_commit();
            };
            const uint32_t hb0 = tc::smem_u32(sH), wn0 = tc::smem_u32(sWn);
            auto issue = [&](uint32_t u, uint32_t tb, bool first) {
                const uint64_t db = tc::umma_desc_k_sw128(tb + u * H_CHUNK);
                const uint32_t a_rz = tmem + A_RZ + u * 32;
                if ((int)u < KC_T) {
                    const uint32_t a_n = tmem + G::A_N + u * 32;
                    if (first) fwd_issue_chunk_ts<true>(tmem, a_rz, a_n, db); else fwd_issue_chunk_ts<false>(tmem, a_rz, a_n, db);
                } else {
                    const uint64_t dw = tc::umma_desc_k_sw128(wn0 + (u - (uint32_t)KC_T) * TAIL_TILE);
                    if (first) fwd_issue_chunk_ss<true>(tmem, a_rz, dw, db); else fwd_issue_chunk_ss<false>(tmem, a_rz, dw, db);
                }
            };
            for (int s = 1; s < T; ++s) {
                const int pb = (s - 1) & 1;
                const uint32_t tb = hb0 + (uint32_t)pb * TILE_BYTES;
                if (ok) ok = tc::mbar_wait(epi_done, epi_rounds & 1, p.dbg, 0x3400 + (s & 0xff));
                ++epi_rounds;
                tc::tcgen05_fence_after();
                issue(c, tb, true);                                        // own chunk first (it is local)
                for (uint32_t i = 1; i < (uint32_t)CS; ++i) {
                    const uint32_t u = (c + i) % CS;
                    if (ok) ok = tc::mbar_wait(&h_full[pb * 8 + u], (pb ? hf_use1 : hf_use0) & 1, p.dbg, 0x3500 + (s & 0xff));
                    if (s + 2 < T) tc::mbar_arrive_expect_tx(&h_full[pb * 8 + u], H_CHUNK);      // h_{s+1} comes to this buffer
                    tc::tcgen05_fence_after();
                    issue(u, tb, false);
                }
                if (pb) ++hf_use1; else ++hf_use0;
                tc::tma_store_wait_read();
                tc::umma_commit(mma_done);
                store_tile(s - 1);
            }
            if (ok) ok = tc::mbar_wait(epi_done, epi_rounds & 1, p.dbg, 0x3400);
            store_tile(T - 1);
            tc::tma_store_wait_all();
        }
    } else {
        // ---- epilogue.  TMEM lane quarter q = warp & 3: q < 2 reads r and n of unit 32q + lane, q >= 2 reads z of unit
        // 32(q-2) + lane; column half = warp >> 2 (16 columns).  After the swap with warp ^ 2 this thread owns unit j, 8 columns.
        const int q = warp & 3, half = warp >> 2, part = q >> 1;
        const int j = (q & 1) * 32 + lane;
        const int unit = (int)c * UNITS + j;
        const int c0 = 16 * half + 8 * part;               // == 8 * (warp >> 1)
        const int tid = threadIdx.x;
        const float bhn = p.b_hn[d * H + unit];
        const bool has_h0 = p.h0 != nullptr && p.gh0 != nullptr;
        float hprev[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) hprev[i] = has_h0 ? p.h0[((int64_t)d * B + tile * NB + c0 + i) * H + unit] : 0.f;
        uint32_t h_off[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) h_off[i] = c * H_CHUNK + tc::sw128_offset(c0 + i, j);
        // the 16-byte piece this lane forwards to the peers: 8 units of lane group lane/8, batch row c0 + lane%8
        const uint32_t fwd_off = c * H_CHUNK + tc::sw128_offset(c0 + (lane & 7), (q & 1) * 32 + (lane >> 3) * 8);
        const uint32_t sIn_u = tc::smem_u32(sIn), sH_u = tc::smem_u32(sH);
        const uint32_t xmine = tc::smem_u32(sX) + (uint32_t)((warp * 4 * 32 + lane) * 16);
        const uint32_t xpeer = tc::smem_u32(sX) + (uint32_t)(((warp ^ 2) * 4 * 32 + lane) * 16);
        bool ok = true;
        uint32_t mma_rounds = 0, xch_rounds = 0;
        for (int s = 0; s < T; ++s) {
            const int t = d == 0 ? s : T - 1 - s;
            const size_t blk = blk_index(d, tile, t, (int)c, ntiles, T, CS);
            float gr[8], gz[8], gn[8];
            {
                const int st = s % NSF;
                if (ok) ok = tc::mbar_wait(&in_full[st], (s / NSF) & 1, p.dbg, 0x3200 + (s & 0xff));
                const uint32_t gp = sIn_u + (uint32_t)st * GI_BLOCK + 16u * tid;
                const uint4 u0 = tc::lds_u4(gp), u1 = tc::lds_u4(gp + 4096), u2 = tc::lds_u4(gp + 8192);
                unpack8(u0, gr); unpack8(u1, gz); unpack8(u2, gn);
            }
            float ar[8], az[8], an[8];
            if (s > 0) {
                if (ok) ok = tc::mbar_wait(mma_done, mma_rounds & 1, p.dbg, 0x3600 + (s & 0xff));
                ++mma_rounds;
                tc::tcgen05_fence_after();
                const uint32_t ta = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(16 * half);
                float va[16], vb[16];
                if (part == 0) {
                    tmem_ld16f(ta + D_RZ, va); tmem_ld16f(ta + D_N, vb);     // r, n of this unit
                    tmem_ld_wait_pin(va, vb);
                    tc::sts_f4(xmine, make_float4(va[8], va[9], va[10], va[11]));
                    tc::sts_f4(xmine + 512, make_float4(va[12], va[13], va[14], va[15]));
                    tc::sts_f4(xmine + 1024, make_float4(vb[8], vb[9], vb[10], vb[11]));
                    tc::sts_f4(xmine + 1536, make_float4(vb[12], vb[13], vb[14], vb[15]));
                } else {
                    tmem_ld16f(ta + D_RZ, va);                                // z of this unit (lanes 64..127)
                    tmem_ld_wait_pin(va);
                    tc::sts_f4(xmine, make_float4(va[0], va[1], va[2], va[3]));
                    tc::sts_f4(xmine + 512, make_float4(va[4], va[5], va[6], va[7]));
                }
                tc::tcgen05_fence_before();
                __syncwarp();
                if (lane == 0) tc::mbar_arrive(&xch[warp]);
                if (ok) ok = tc::mbar_wait(&xch[warp ^ 2], xch_rounds & 1, p.dbg, 0x3900 + (s & 0xff));
                ++xch_rounds;
                if (part == 0) {
                    const float4 z0 = tc::lds_f4(xpeer), z1 = tc::lds_f4(xpeer + 512);
                    az[0] = z0.x; az[1] = z0.y; az[2] = z0.z; az[3] = z0.w; az[4] = z1.x; az[5] = z1.y; az[6] = z1.z; az[7] = z1.w;
#pragma unroll
                    for (int i = 0; i < 8; ++i) { ar[i] = va[i]; an[i] = vb[i]; }
                } else {
                    const float4 r0 = tc::lds_f4(xpeer), r1 = tc::lds_f4(xpeer + 512), n0 = tc::lds_f4(xpeer + 1024), n1 = tc::lds_f4(xpeer + 1536);
                    ar[0] = r0.x; ar[1] = r0.y; ar[2] = r0.z; ar[3] = r0.w; ar[4] = r1.x; ar[5] = r1.y; ar[6] = r1.z; ar[7] = r1.w;
                    an[0] = n0.x; an[1] = n0.y; an[2] = n0.z; an[3] = n0.w; an[4] = n1.x; an[5] = n1.y; an[6] = n1.z; an[7] = n1.w;
#pragma unroll
                    for (int i = 0; i < 8; ++i) az[i] = va[8 + i];
                }
            } else if (has_h0) {
                // step 0 with an initial state: the recurrent product W_hh h0 comes from the caller (no MMA at step 0)
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const float* gp = p.gh0 + ((int64_t)d * B + tile * NB + c0 + i) * 3 * H + unit;
                    ar[i] = gp[0]; az[i] = gp[H]; an[i] = gp[2 * H];
                }
            } else {
#pragma unroll
                for (int i = 0; i < 8; ++i) { ar[i] = 0.f; az[i] = 0.f; an[i] = 0.f; }
            }
            float r8[8], z8[8], n8[8], hn8[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float r = tcs::sigmoid_fast(gr[i] + ar[i]);
                const float z = tcs::sigmoid_fast(gz[i] + az[i]);
                hn8[i] = an[i] + bhn;
                const float n = tcs::tanh_fast(fmaf(r, hn8[i], gn[i]));
                r8[i] = r; z8[i] = z; n8[i] = n;
                hprev[i] = fmaf(z, hprev[i] - n, n);
            }
            {   // publish h (bf16) in this CTA's chunk of operand buffer s & 1, forward it to the peers, one arrival per warp
                const uint32_t hb = sH_u + (uint32_t)(s & 1) * TILE_BYTES;
#pragma unroll
                for (int i = 0; i < 8; ++i) tc::sts_bf16(hb + h_off[i], __float2bfloat16(hprev[i]));
                tc::tcgen05_fence_before();
                if (s + 1 < T) {
                    __syncwarp();
                    const uint32_t a_h = hb + fwd_off, a_bar = tc::smem_u32(&h_full[(s & 1) * 8 + (int)c]);
                    const uint4 vh = tc::lds_u4(a_h);
#pragma unroll
                    for (uint32_t i = 1; i < (uint32_t)CS; ++i) {
                        const uint32_t pr = (c + i) % CS;
                        tc::st_async_v4(tc::mapa_u32(a_h, pr), vh, tc::mapa_u32(a_bar, pr));
                    }
                }
                tc::fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) tc::mbar_arrive(epi_done);
                // the ring slot is released only here: the published h depends on every value loaded from it (see tc_scan.cuh)
                if (lane == 0) tc::mbar_arrive(&in_empty[s % NSF]);
            }
            {   // stash (off the chain)
                uint4* gs = reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(p.GW) + blk * G_BLOCK) + tid;
                gs[0] = pack8(r8); gs[256] = pack8(z8); gs[512] = pack8(n8); gs[768] = pack8(hn8);
                uint4* ys = reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(p.YBW) + blk * YB_BLOCK) + tid;
                ys[0] = pack8(hprev);
            }
            if (s == T - 1 && p.hn_out) {
#pragma unroll
                for (int i = 0; i < 8; ++i) p.hn_out[((int64_t)d * B + tile * NB + c0 + i) * H + unit] = hprev[i];
            }
        }
    }
    tc::tcgen05_fence_before();
    __syncthreads();
    tc::cluster_sync_all();
    if (warp == EPI_WARPS) tc::tmem_dealloc(tmem, 512);
}

static inline cudaError_t launch_fwd(const FwdParams& p_in, cudaStream_t st) {
    FwdParams p = p_in;
    if (p.H != 512 || p.B % NB != 0) return cudaErrorInvalidValue;
    // (a ping-pong form of this kernel - the two warp groups decoupled per 16-row sub-tile like the backward below - was built and
    // measured SLOWER, 9.97 vs 5.9 us/step: the control thread serves the sub-tiles in order and each waits for seven peers' chunks)
    {
        const uint64_t dims[2] = {(uint64_t)p.D * p.H, (uint64_t)p.T * p.B};
        const uint64_t strides[1] = {(uint64_t)p.D * p.H * 2};
        const uint32_t box[2] = {64u, (uint32_t)NB};
        if (make_tmap_bf16(&p.tmY, p.Yrow, 2, dims, strides, box) != 0) return cudaErrorInvalidValue;
    }
    const int CS = p.H / UNITS;
    const size_t smem = fwd_smem_bytes(p.H);
    void (*kern)(FwdParams) = gru_scanw_fwd_kernel<512>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
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

// =================================================================================================
// Backward scan (BPTT), reduction-partitioned (see the header comment and tc_scan_x.cuh).
//   A operand (TMEM): lane i of row block rb holds W_hh[q][k] for k = 128*rb + i and the CTA's own gate rows
//   q = g*H + 64c + jj, K index kq = g*64 + jj (192 = 12 K-steps): image [D][CS][128 lanes][NRB*192].
//   B operand (smem): this CTA's dgh tile [32 x 192] (da_r | da_z | da_n*r of its 64 units).
//   D[rb] (32 columns each): partial dh for output unit k; partials of units owned by another CTA travel to its receive
//   buffer, the owner adds the CS contributions.
// =================================================================================================
struct BwdParams {
    int B, T, H, D;
    const __nv_bfloat16* WTimg;
    const __nv_bfloat16* GW;
    const __nv_bfloat16* YBW;
    const float* dYBW;              // lower layers
    const float* h0;                // nullable [D][B][H]: h_prev of the first forward step
    float* dh0;                     // nullable [D][B][H]: gradient of the initial hidden state
    const float* dlogits;           // top layer: dL/dlogits [B][C], head weights and the max-pool arg-max (see tc_scan.cuh)
    const float* lin_w;
    const int* arg;
    int C;
    __nv_bfloat16* dgi_row;         // [R][D*3H]
    __nv_bfloat16* dghn_row;        // [R][D*H]
    CUtensorMap tmGI, tmGN;
    float* db_ih;
    float* db_hh;
    int64_t dir_stride;
    unsigned int* dbg;
};

__device__ __forceinline__ void bwd_issue_block(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc) {
    constexpr uint32_t idesc = tc::umma_idesc_bf16(128, NB);
#pragma unroll
    for (int g = 0; g < 3; ++g) {
#pragma unroll
        for (int kk = 0; kk < 4; ++kk)
            tcs::umma_bf16_ts(tmem_d, tmem_a + (uint32_t)((g * 4 + kk) * 8), desc + (uint64_t)(g * (H_CHUNK >> 4) + 2 * kk), idesc,
                              (g == 0 && kk == 0) ? 0u : 1u);
    }
}

template <int H>
__global__ void __launch_bounds__(THREADS, 1) gru_scanw_bwd_kernel(const __grid_constant__ BwdParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    using G = Geo<H>;
    constexpr int CS = G::CS, NRB = G::NRB, RECV_BYTES = G::RECV_BYTES;
    constexpr int DT_BYTES = 3 * H_CHUNK;                 // one dgh tile
    constexpr uint32_t A_COL = NRB * NB;                   // accumulators in columns [0, NRB*32), weights behind them (NRB*96 columns)
    const int B = p.B, T = p.T;
    uint8_t* sD = smem;                                    // [2 buf][3 gates][H_CHUNK]
    uint8_t* sN = sD + (size_t)2 * DT_BYTES;               // [2 buf][H_CHUNK]   da_n (dgi n-gate rows, store only)
    uint8_t* sR = sN + (size_t)2 * H_CHUNK;                // [2 buf][CS src][8 cg][64 j] float4
    uint8_t* sIn = sR + (size_t)2 * RECV_BYTES;            // [NSB][G | YB | dY]
    uint64_t* bars = reinterpret_cast<uint64_t*>(sIn + (size_t)NSB * BWD_STAGE);
    uint64_t* recv_full = bars;        // [2]
    uint64_t* mma_a = bars + 2;        // the row blocks owned by other CTA pairs are done
    uint64_t* mma_b = bars + 3;        // all row blocks done
    uint64_t* epi_done = bars + 4;
    uint64_t* st_done = bars + 5;
    uint64_t* in_full = bars + 6;      // [NSB]
    uint64_t* in_empty = bars + 6 + NSB;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 6 + 2 * NSB);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t c = tc::cluster_ctarank();
    const int cluster_id = blockIdx.x / CS;
    const int ntiles = B / NB;
    const int d = cluster_id / ntiles, tile = cluster_id % ntiles;
    const bool top = p.dlogits != nullptr;
    const int rb_own = (int)c >> 1;                        // row block that contains this CTA's own units

    if (threadIdx.x == 0) {
        tc::mbar_init(&recv_full[0], 1);
        tc::mbar_init(&recv_full[1], 1);
        tc::mbar_init(mma_a, 1);
        tc::mbar_init(mma_b, 1);
        tc::mbar_init(epi_done, EPI_WARPS);
        tc::mbar_init(st_done, EPI_WARPS);
        for (int i = 0; i < NSB; ++i) { tc::mbar_init(&in_full[i], 1); tc::mbar_init(&in_empty[i], EPI_WARPS); }
        tc::fence_mbar_init();
    }
    if (warp == EPI_WARPS) tc::tmem_alloc(tmem_slot, 512);
    tc::tcgen05_fence_before();
    __syncthreads();
    tc::cluster_sync_all();
    tc::tcgen05_fence_after();
    const uint32_t tmem = *tmem_slot;
    if (warp < EPI_WARPS)
        tcs::load_weights_to_tmem(p.WTimg + ((size_t)d * CS + c) * 128 * (NRB * 192), NRB * 192, tmem, A_COL, warp, lane);
    tc::tcgen05_fence_before();
    __syncthreads();
    tc::tcgen05_fence_after();

    if (warp == EPI_WARPS + 1) {
        if (tc::elect_one()) {
            bool ok = true;
            for (int s = 0; s < T; ++s) {
                const int st = s % NSB;
                if (s >= NSB && ok) ok = tc::mbar_wait(&in_empty[st], ((s / NSB) - 1) & 1, p.dbg, 0x4300 + (s & 0xff));
                const int t = d == 0 ? T - 1 - s : s;
                const bool first = d == 0 ? t == 0 : t == T - 1;
                uint8_t* dst = sIn + (size_t)st * BWD_STAGE;
                tc::mbar_arrive_expect_tx(&in_full[st], (uint32_t)(G_BLOCK + (top ? 0 : DY_BLOCK) + (first ? 0 : YB_BLOCK)));
                const size_t blk = blk_index(d, tile, t, (int)c, ntiles, T, CS);
                tc::bulk_g2s(dst, reinterpret_cast<const uint8_t*>(p.GW) + blk * G_BLOCK, G_BLOCK, &in_full[st]);
                if (!top) tc::bulk_g2s(dst + G_BLOCK + YB_BLOCK, reinterpret_cast<const uint8_t*>(p.dYBW) + blk * DY_BLOCK, DY_BLOCK, &in_full[st]);
                if (!first) {
                    const size_t pblk = blk_index(d, tile, d == 0 ? t - 1 : t + 1, (int)c, ntiles, T, CS);
                    tc::bulk_g2s(dst + G_BLOCK, reinterpret_cast<const uint8_t*>(p.YBW) + pblk * YB_BLOCK, YB_BLOCK, &in_full[st]);
                }
            }
        }
    } else if (warp == EPI_WARPS) {
        if (tc::elect_one()) {
            bool ok = true;
            auto store_tile = [&](int step) {
                const int tt = d == 0 ? T - 1 - step : step;
                const int row = tt * B + tile * NB;
                const uint8_t* tb = sD + (size_t)(step & 1) * DT_BYTES;
                const uint8_t* nb = sN + (size_t)(step & 1) * H_CHUNK;
                const int cu = (int)c * UNITS;
                tc::tma_store_2d(&p.tmGI, tb, d * 3 * H + cu, row);                               // da_r
                tc::tma_store_2d(&p.tmGI, tb + H_CHUNK, d * 3 * H + H + cu, row);                 // da_z
                tc::tma_store_2d(&p.tmGI, nb, d * 3 * H + 2 * H + cu, row);                       // da_n
                tc::tma_store_2d(&p.tmGN, tb + 2 * H_CHUNK, d * H + cu, row);                     // da_n * r
                tc::tma_store_commit();
            };
            const uint32_t db0 = tc::smem_u32(sD);
            const int Tend = T + (p.dh0 ? 1 : 0);          // one more product (no gate math) when d(h0) is wanted
            for (int s = 1; s < Tend; ++s) {
                const int pb = (s - 1) & 1;
                if (ok) ok = tc::mbar_wait(epi_done, (s - 1) & 1, p.dbg, 0x4700 + (s & 0xff));
                tc::tcgen05_fence_after();
                tc::mbar_arrive_expect_tx(&recv_full[s & 1], (uint32_t)(CS - 1) * 8192u);
                const uint64_t dd = tc::umma_desc_k_sw128(db0 + (uint32_t)pb * DT_BYTES);
#pragma unroll
                for (int i = 1; i < NRB; ++i) {
                    const int rb = (rb_own + i) % NRB;
                    bwd_issue_block(tmem + (uint32_t)(rb * NB), tmem + A_COL + (uint32_t)(rb * 96), dd);
                }
                tc::umma_commit(mma_a);
                bwd_issue_block(tmem + (uint32_t)(rb_own * NB), tmem + A_COL + (uint32_t)(rb_own * 96), dd);
                tc::tma_store_wait_read();
                tc::umma_commit(mma_b);
                if (ok) ok = tc::mbar_wait(st_done, (s - 1) & 1, p.dbg, 0x4a00 + (s & 0xff));
                store_tile(s - 1);
            }
            if (Tend == T) {
                if (ok) ok = tc::mbar_wait(epi_done, (T - 1) & 1, p.dbg, 0x4700);
                if (ok) ok = tc::mbar_wait(st_done, (T - 1) & 1, p.dbg, 0x4a00);
                store_tile(T - 1);
            }
            tc::tma_store_wait_all();
        }
    } else {
        // ---- epilogue.  Owner role: unit j = (warp & 1)*32 + lane of this CTA, batch columns [8*(warp >> 1), +8).
        //      Partial-sum role: TMEM lane quarter q = warp & 3 -> output unit k = 128*rb + 32q + lane, columns [16*half, +16).
        const int q = warp & 3, half = warp >> 2;
        const int j = (warp & 1) * 32 + lane;
        const int unit = (int)c * UNITS + j;
        const int c0 = 8 * (warp >> 1);
        const int tid = threadIdx.x;
        float dhz[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) dhz[i] = 0.f;
        float h_avg[8], h_max[8];
        int h_arg[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) { h_avg[i] = 0.f; h_max[i] = 0.f; h_arg[i] = -1; }
        if (top) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int b = tile * NB + c0 + i;
                float dl = 0.f, dm = 0.f, da = 0.f;
                for (int cc = 0; cc < p.C; ++cc) {
                    const float g = p.dlogits[(int64_t)b * p.C + cc];
                    const float* w = p.lin_w + (int64_t)cc * 3 * H;
                    dl = fmaf(g, w[unit], dl); dm = fmaf(g, w[H + unit], dm); da = fmaf(g, w[2 * H + unit], da);
                }
                dhz[i] = dl;
                h_avg[i] = da / (float)T; h_max[i] = dm; h_arg[i] = p.arg[(int64_t)b * H + unit];
            }
        }
        float sb_r = 0.f, sb_z = 0.f, sb_n = 0.f, sb_nr = 0.f;
        uint32_t e_off[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) e_off[i] = tc::sw128_offset(c0 + i, j);
        // partial-sum destination inside a receive buffer: [src = c][cg = 4*half + i][jd] float4, jd = (q & 1)*32 + lane
        const uint32_t r_off = (((uint32_t)c * 8 + 4 * half) * 64 + (uint32_t)((q & 1) * 32 + lane)) * 16;
        const uint32_t sIn_u = tc::smem_u32(sIn), sR_u = tc::smem_u32(sR), sD_u = tc::smem_u32(sD), sN_u = tc::smem_u32(sN);
        bool ok = true;
        auto reduce_partials = [&](int s, float (&acc)[8]) {
            const int buf = s & 1;
            const uint32_t rb_local = sR_u + (uint32_t)buf * RECV_BYTES;
            const uint32_t rbar_l = tc::smem_u32(&recv_full[buf]);
            auto route = [&](int rb) {
                float v[16];
                tmem_ld16f(tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(rb * NB + 16 * half), v);
                tmem_ld_wait_pin(v);
                const uint32_t dest = (uint32_t)(2 * rb + (q >> 1));
                const uint32_t lp = rb_local + r_off;
                if (dest == c) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) tc::sts_f4(lp + (uint32_t)(i * 64 * 16), make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]));
                } else {
                    const uint32_t ra = tc::mapa_u32(lp, dest), rbr = tc::mapa_u32(rbar_l, dest);
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        uint4 u;
                        u.x = __float_as_uint(v[4 * i]); u.y = __float_as_uint(v[4 * i + 1]); u.z = __float_as_uint(v[4 * i + 2]); u.w = __float_as_uint(v[4 * i + 3]);
                        tc::st_async_v4(ra + (uint32_t)(i * 64 * 16), u, rbr);
                    }
                }
            };
            if (ok) ok = tc::mbar_wait(mma_a, (s - 1) & 1, p.dbg, 0x4800 + (s & 0xff));
            tc::tcgen05_fence_after();
#pragma unroll
            for (int i = 1; i < NRB; ++i) route((rb_own + i) % NRB);
            if (ok) ok = tc::mbar_wait(mma_b, (s - 1) & 1, p.dbg, 0x4900 + (s & 0xff));
            tc::tcgen05_fence_after();
            route(rb_own);
            tc::tcgen05_fence_before();
            epi_barrier();                                   // this CTA's own contributions are in the buffer
            if (ok) ok = tc::mbar_wait_cluster(&recv_full[buf], ((s - 1) >> 1) & 1, p.dbg, 0x4b00 + (s & 0xff));
#pragma unroll
            for (int i = 0; i < 8; ++i) acc[i] = 0.f;
#pragma unroll
            for (int src = 0; src < CS; ++src) {
                const uint32_t rp = rb_local + (uint32_t)((((src * 8 + 2 * (warp >> 1)) * 64) + j) * 16);
                const float4 x0 = tc::lds_f4(rp), x1 = tc::lds_f4(rp + 64 * 16);
                acc[0] += x0.x; acc[1] += x0.y; acc[2] += x0.z; acc[3] += x0.w; acc[4] += x1.x; acc[5] += x1.y; acc[6] += x1.z; acc[7] += x1.w;
            }
        };
        for (int s = 0; s < T; ++s) {
            const int t = d == 0 ? T - 1 - s : s;
            const bool first = d == 0 ? t == 0 : t == T - 1;
            float vr[8], vz[8], vn[8], vhn[8], vhp[8], vdy[8];
            {
                const int st = s % NSB;
                if (ok) ok = tc::mbar_wait(&in_full[st], (s / NSB) & 1, p.dbg, 0x4200 + (s & 0xff));
                const uint32_t gp = sIn_u + (uint32_t)st * BWD_STAGE + 16u * tid;
                const uint4 u0 = tc::lds_u4(gp), u1 = tc::lds_u4(gp + 4096), u2 = tc::lds_u4(gp + 8192), u3 = tc::lds_u4(gp + 12288);
                uint4 uh = make_uint4(0u, 0u, 0u, 0u);
                float4 y0 = make_float4(0.f, 0.f, 0.f, 0.f), y1 = y0;
                if (!first) uh = tc::lds_u4(gp + G_BLOCK);
                if (!top) { y0 = tc::lds_f4(sIn_u + (uint32_t)st * BWD_STAGE + G_BLOCK + YB_BLOCK + 32u * tid); y1 = tc::lds_f4(sIn_u + (uint32_t)st * BWD_STAGE + G_BLOCK + YB_BLOCK + 32u * tid + 16); }
                unpack8(u0, vr); unpack8(u1, vz); unpack8(u2, vn); unpack8(u3, vhn); unpack8(uh, vhp);
                if (first && p.h0) {                        // the caller's initial state, in fp32
#pragma unroll
                    for (int i = 0; i < 8; ++i) vhp[i] = p.h0[((int64_t)d * B + tile * NB + c0 + i) * H + unit];
                }
                vdy[0] = y0.x; vdy[1] = y0.y; vdy[2] = y0.z; vdy[3] = y0.w; vdy[4] = y1.x; vdy[5] = y1.y; vdy[6] = y1.z; vdy[7] = y1.w;
                if (top) {
#pragma unroll
                    for (int i = 0; i < 8; ++i) vdy[i] = h_avg[i] + (h_arg[i] == t ? h_max[i] : 0.f);
                }
            }
            float c_n[8], c_r[8], c_z[8], pre[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float r = vr[i], z = vz[i], n = vn[i];
                c_n[i] = (1.f - z) * (1.f - n * n);
                c_r[i] = vhn[i] * r * (1.f - r);
                c_z[i] = (vhp[i] - n) * z * (1.f - z);
                pre[i] = dhz[i] + vdy[i];
            }
            float acc[8];
            const int buf = s & 1;
            if (s > 0) reduce_partials(s, acc);
            else {
#pragma unroll
                for (int i = 0; i < 8; ++i) acc[i] = 0.f;
            }
            const uint32_t tileb = sD_u + (uint32_t)buf * DT_BYTES;
            const uint32_t nbuf = sN_u + (uint32_t)buf * H_CHUNK;
            float dar[8], daz[8], dan[8], danr[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float dh = acc[i] + pre[i];
                dan[i] = dh * c_n[i];
                dar[i] = dan[i] * c_r[i];
                daz[i] = dh * c_z[i];
                danr[i] = dan[i] * vr[i];
                dhz[i] = dh * vz[i];
                tc::sts_bf16(tileb + e_off[i], __float2bfloat16(dar[i]));
                tc::sts_bf16(tileb + H_CHUNK + e_off[i], __float2bfloat16(daz[i]));
                tc::sts_bf16(tileb + 2 * H_CHUNK + e_off[i], __float2bfloat16(danr[i]));
            }
            tc::tcgen05_fence_before();
            tc::fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(epi_done);
            // the ring slot is released only here: the published dgh depends on every value loaded from it (see tc_scan.cuh)
            if (lane == 0) tc::mbar_arrive(&in_empty[s % NSB]);
#pragma unroll
            for (int i = 0; i < 8; ++i) tc::sts_bf16(nbuf + e_off[i], __float2bfloat16(dan[i]));
            tc::fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(st_done);
#pragma unroll
            for (int i = 0; i < 8; ++i) { sb_r += dar[i]; sb_z += daz[i]; sb_n += dan[i]; sb_nr += danr[i]; }
        }
        float* dbi = p.db_ih + (int64_t)d * p.dir_stride;
        float* dbh = p.db_hh + (int64_t)d * p.dir_stride;
        atomicAdd(dbi + unit, sb_r); atomicAdd(dbi + H + unit, sb_z); atomicAdd(dbi + 2 * H + unit, sb_n);
        atomicAdd(dbh + unit, sb_r); atomicAdd(dbh + H + unit, sb_z); atomicAdd(dbh + 2 * H + unit, sb_nr);
        if (p.dh0) {
            // gradient of the initial hidden state = z-carry of the last step + W_hh^T dgh of the last step (one more product)
            float acc[8];
            reduce_partials(T, acc);
#pragma unroll
            for (int i = 0; i < 8; ++i) p.dh0[((int64_t)d * B + tile * NB + c0 + i) * H + unit] = dhz[i] + acc[i];
        }
    }
    tc::tcgen05_fence_before();
    __syncthreads();
    tc::cluster_sync_all();
    if (warp == EPI_WARPS) tc::tmem_dealloc(tmem, 512);
}

// ping-pong form: a 16-row dgh sub-tile against one row block: 12 MMAs with N = 16
__device__ __forceinline__ void bwd2_issue_block(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc) {
    constexpr uint32_t idesc = tc::umma_idesc_bf16(128, tcx::NBS);
#pragma unroll
    for (int g = 0; g < 3; ++g) {
#pragma unroll
        for (int kk = 0; kk < 4; ++kk)
            tcs::umma_bf16_ts(tmem_d, tmem_a + (uint32_t)((g * 4 + kk) * 8), desc + (uint64_t)(g * (tcx::HS_CHUNK >> 4) + 2 * kk), idesc,
                              (g == 0 && kk == 0) ? 0u : 1u);
    }
}

template <int H>
__global__ void __launch_bounds__(THREADS, 1) gru_scanw_bwd2_kernel(const __grid_constant__ BwdParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    using G = Geo<H>;
    constexpr int CS = G::CS, NRB = G::NRB, RECV_BYTES = G::RECV_BYTES;
    // Ping-pong form (see tcx::gru_scanx_bwd2_kernel): epilogue warps 0-3 only ever touch batch columns 0-15, warps 4-7 columns
    // 16-31, so the two warp groups run as two decoupled 16-row sub-tiles (own dgh tiles with N = 16, accumulators, barriers).
    constexpr int NBS = tcx::NBS, HS_CHUNK = tcx::HS_CHUNK;
    constexpr int DT_BYTES = 3 * HS_CHUNK;                // one dgh sub-tile
    constexpr int SUBD = 2 * DT_BYTES, SUBN = 2 * HS_CHUNK;
    constexpr uint32_t A_COL = NRB * NB;                   // accumulators in columns [0, NRB*32): [sub][rb][16]; weights behind them
    const int B = p.B, T = p.T;
    uint8_t* sD = smem;                                    // [2 sub][2 buf][3 gates][HS_CHUNK]
    uint8_t* sN = sD + (size_t)2 * SUBD;                   // [2 sub][2 buf][HS_CHUNK]   da_n (dgi n-gate rows, store only)
    uint8_t* sR = sN + (size_t)2 * SUBN;                   // [2 buf][CS src][8 cg][64 j] float4 (column groups 0-3: sub-tile 0, 4-7: sub-tile 1)
    uint8_t* sIn = sR + (size_t)2 * RECV_BYTES;            // [NSB][G | YB | dY]
    uint64_t* bars = reinterpret_cast<uint64_t*>(sIn + (size_t)NSB * BWD_STAGE);
    uint64_t* recv_full = bars;        // [2 sub][2 buf]
    uint64_t* mma_a = bars + 4;        // [2 sub] the row blocks owned by other CTA pairs are done
    uint64_t* mma_b = bars + 6;        // [2 sub] all row blocks done
    uint64_t* epi_done = bars + 8;     // [2 sub]
    uint64_t* st_done = bars + 10;     // [2 sub]
    uint64_t* in_full = bars + 12;     // [NSB]
    uint64_t* in_empty = bars + 12 + NSB;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 12 + 2 * NSB);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t c = tc::cluster_ctarank();
    const int cluster_id = blockIdx.x / CS;
    const int ntiles = B / NB;
    const int d = cluster_id / ntiles, tile = cluster_id % ntiles;
    const bool top = p.dlogits != nullptr;
    const int rb_own = (int)c >> 1;                        // row block that contains this CTA's own units

    if (threadIdx.x == 0) {
        for (int i = 0; i < 4; ++i) tc::mbar_init(&recv_full[i], 1);
        for (int i = 0; i < 2; ++i) {
            tc::mbar_init(&mma_a[i], 1); tc::mbar_init(&mma_b[i], 1);
            tc::mbar_init(&epi_done[i], EPI_WARPS / 2); tc::mbar_init(&st_done[i], EPI_WARPS / 2);
        }
        for (int i = 0; i < NSB; ++i) { tc::mbar_init(&in_full[i], 1); tc::mbar_init(&in_empty[i], EPI_WARPS); }
        tc::fence_mbar_init();
    }
    if (warp == EPI_WARPS) tc::tmem_alloc(tmem_slot, 512);
    tc::tcgen05_fence_before();
    __syncthreads();
    tc::cluster_sync_all();
    tc::tcgen05_fence_after();
    const uint32_t tmem = *tmem_slot;
    if (warp < EPI_WARPS)
        tcs::load_weights_to_tmem(p.WTimg + ((size_t)d * CS + c) * 128 * (NRB * 192), NRB * 192, tmem, A_COL, warp, lane);
    tc::tcgen05_fence_before();
    __syncthreads();
    tc::tcgen05_fence_after();

    if (warp == EPI_WARPS + 1) {
        if (tc::elect_one()) {
            bool ok = true;
            for (int s = 0; s < T; ++s) {
                const int st = s % NSB;
                if (s >= NSB && ok) ok = tc::mbar_wait(&in_empty[st], ((s / NSB) - 1) & 1, p.dbg, 0x4300 + (s & 0xff));
                const int t = d == 0 ? T - 1 - s : s;
                const bool first = d == 0 ? t == 0 : t == T - 1;
                uint8_t* dst = sIn + (size_t)st * BWD_STAGE;
                tc::mbar_arrive_expect_tx(&in_full[st], (uint32_t)(G_BLOCK + (top ? 0 : DY_BLOCK) + (first ? 0 : YB_BLOCK)));
                const size_t blk = blk_index(d, tile, t, (int)c, ntiles, T, CS);
                tc::bulk_g2s(dst, reinterpret_cast<const uint8_t*>(p.GW) + blk * G_BLOCK, G_BLOCK, &in_full[st]);
                if (!top) tc::bulk_g2s(dst + G_BLOCK + YB_BLOCK, reinterpret_cast<const uint8_t*>(p.dYBW) + blk * DY_BLOCK, DY_BLOCK, &in_full[st]);
                if (!first) {
                    const size_t pblk = blk_index(d, tile, d == 0 ? t - 1 : t + 1, (int)c, ntiles, T, CS);
                    tc::bulk_g2s(dst + G_BLOCK, reinterpret_cast<const uint8_t*>(p.YBW) + pblk * YB_BLOCK, YB_BLOCK, &in_full[st]);
                }
            }
        }
    } else if (warp == EPI_WARPS) {
        if (tc::elect_one()) {
            bool ok = true;
            auto store_tile = [&](int sub, int step) {        // 16-row boxes (the tensor maps of this form have box 64 x 16)
                const int tt = d == 0 ? T - 1 - step : step;
                const int row = tt * B + tile * NB + sub * NBS;
                const uint8_t* tb = sD + (size_t)sub * SUBD + (size_t)(step & 1) * DT_BYTES;
                const uint8_t* nb = sN + (size_t)sub * SUBN + (size_t)(step & 1) * HS_CHUNK;
                const int cu = (int)c * UNITS;
                tc::tma_store_2d(&p.tmGI, tb, d * 3 * H + cu, row);                               // da_r
                tc::tma_store_2d(&p.tmGI, tb + HS_CHUNK, d * 3 * H + H + cu, row);                // da_z
                tc::tma_store_2d(&p.tmGI, nb, d * 3 * H + 2 * H + cu, row);                       // da_n
                tc::tma_store_2d(&p.tmGN, tb + 2 * HS_CHUNK, d * H + cu, row);                    // da_n * r
                tc::tma_store_commit();
            };
            const uint32_t db0 = tc::smem_u32(sD);
            const int Tend = T + (p.dh0 ? 1 : 0);          // one more product (no gate math) when d(h0) is wanted
            for (int s = 1; s < Tend; ++s) {
                const int pb = (s - 1) & 1;
#pragma unroll
                for (int sub = 0; sub < 2; ++sub) {
                    if (ok) ok = tc::mbar_wait(&epi_done[sub], (s - 1) & 1, p.dbg, 0x4700 + (s & 0xff));
                    tc::tcgen05_fence_after();
                    tc::mbar_arrive_expect_tx(&recv_full[sub * 2 + (s & 1)], (uint32_t)(CS - 1) * 4096u);
                    const uint64_t dd = tc::umma_desc_k_sw128(db0 + (uint32_t)sub * SUBD + (uint32_t)pb * DT_BYTES);
                    const uint32_t td = tmem + (uint32_t)(sub * NRB * NBS);
#pragma unroll
                    for (int i = 1; i < NRB; ++i) {
                        const int rb = (rb_own + i) % NRB;
                        bwd2_issue_block(td + (uint32_t)(rb * NBS), tmem + A_COL + (uint32_t)(rb * 96), dd);
                    }
                    tc::umma_commit(&mma_a[sub]);
                    bwd2_issue_block(td + (uint32_t)(rb_own * NBS), tmem + A_COL + (uint32_t)(rb_own * 96), dd);
                    tcx::tma_store_wait_read1();       // the tile of THIS sub-tile stored two steps ago has been read
                    tc::umma_commit(&mma_b[sub]);
                    if (ok) ok = tc::mbar_wait(&st_done[sub], (s - 1) & 1, p.dbg, 0x4a00 + (s & 0xff));
                    store_tile(sub, s - 1);
                }
            }
            if (Tend == T) {
                for (int sub = 0; sub < 2; ++sub) {
                    if (ok) ok = tc::mbar_wait(&epi_done[sub], (T - 1) & 1, p.dbg, 0x4700);
                    if (ok) ok = tc::mbar_wait(&st_done[sub], (T - 1) & 1, p.dbg, 0x4a00);
                    store_tile(sub, T - 1);
                }
            }
            tc::tma_store_wait_all();
        }
    } else {
        // ---- epilogue.  Owner role: unit j = (warp & 1)*32 + lane of this CTA, batch columns [8*(warp >> 1), +8).
        //      Partial-sum role: TMEM lane quarter q = warp & 3 -> output unit k = 128*rb + 32q + lane, columns [16*half, +16).
        const int q = warp & 3, half = warp >> 2;          // half == sub-tile of this warp (router AND owner roles)
        const int sub = half;
        const int j = (warp & 1) * 32 + lane;
        const int unit = (int)c * UNITS + j;
        const int c0 = 8 * (warp >> 1);
        const int tid = threadIdx.x;
        float dhz[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) dhz[i] = 0.f;
        float h_avg[8], h_max[8];
        int h_arg[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) { h_avg[i] = 0.f; h_max[i] = 0.f; h_arg[i] = -1; }
        if (top) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int b = tile * NB + c0 + i;
                float dl = 0.f, dm = 0.f, da = 0.f;
                for (int cc = 0; cc < p.C; ++cc) {
                    const float g = p.dlogits[(int64_t)b * p.C + cc];
                    const float* w = p.lin_w + (int64_t)cc * 3 * H;
                    dl = fmaf(g, w[unit], dl); dm = fmaf(g, w[H + unit], dm); da = fmaf(g, w[2 * H + unit], da);
                }
                dhz[i] = dl;
                h_avg[i] = da / (float)T; h_max[i] = dm; h_arg[i] = p.arg[(int64_t)b * H + unit];
            }
        }
        float sb_r = 0.f, sb_z = 0.f, sb_n = 0.f, sb_nr = 0.f;
        uint32_t e_off[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) e_off[i] = tc::sw128_offset(c0 - 16 * sub + i, j);      // row inside the 16-row sub-tile
        // partial-sum destination inside a receive buffer: [src = c][cg = 4*half + i][jd] float4, jd = (q & 1)*32 + lane
        const uint32_t r_off = (((uint32_t)c * 8 + 4 * half) * 64 + (uint32_t)((q & 1) * 32 + lane)) * 16;
        const uint32_t sIn_u = tc::smem_u32(sIn), sR_u = tc::smem_u32(sR), sD_u = tc::smem_u32(sD), sN_u = tc::smem_u32(sN);
        bool ok = true;
        auto reduce_partials = [&](int s, float (&acc)[8]) {
            const int buf = s & 1;
            const uint32_t rb_local = sR_u + (uint32_t)buf * RECV_BYTES;
            const uint32_t rbar_l = tc::smem_u32(&recv_full[sub * 2 + buf]);
            auto route = [&](int rb) {
                float v[16];
                tmem_ld16f(tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(sub * NRB * NBS + rb * NBS), v);
                tmem_ld_wait_pin(v);
                const uint32_t dest = (uint32_t)(2 * rb + (q >> 1));
                const uint32_t lp = rb_local + r_off;
                if (dest == c) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) tc::sts_f4(lp + (uint32_t)(i * 64 * 16), make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]));
                } else {
                    const uint32_t ra = tc::mapa_u32(lp, dest), rbr = tc::mapa_u32(rbar_l, dest);
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        uint4 u;
                        u.x = __float_as_uint(v[4 * i]); u.y = __float_as_uint(v[4 * i + 1]); u.z = __float_as_uint(v[4 * i + 2]); u.w = __float_as_uint(v[4 * i + 3]);
                        tc::st_async_v4(ra + (uint32_t)(i * 64 * 16), u, rbr);
                    }
                }
            };
            if (ok) ok = tc::mbar_wait(&mma_a[sub], (s - 1) & 1, p.dbg, 0x4800 + (s & 0xff));
            tc::tcgen05_fence_after();
#pragma unroll
            for (int i = 1; i < NRB; ++i) route((rb_own + i) % NRB);
            if (ok) ok = tc::mbar_wait(&mma_b[sub], (s - 1) & 1, p.dbg, 0x4900 + (s & 0xff));
            tc::tcgen05_fence_after();
            route(rb_own);
            tc::tcgen05_fence_before();
            asm volatile("bar.sync %0, 128;" ::"r"(1 + sub) : "memory");      // this warp group's own contributions are in the buffer
            if (ok) ok = tc::mbar_wait_cluster(&recv_full[sub * 2 + buf], ((s - 1) >> 1) & 1, p.dbg, 0x4b00 + (s & 0xff));
#pragma unroll
            for (int i = 0; i < 8; ++i) acc[i] = 0.f;
#pragma unroll
            for (int src = 0; src < CS; ++src) {
                const uint32_t rp = rb_local + (uint32_t)((((src * 8 + 2 * (warp >> 1)) * 64) + j) * 16);
                const float4 x0 = tc::lds_f4(rp), x1 = tc::lds_f4(rp + 64 * 16);
                acc[0] += x0.x; acc[1] += x0.y; acc[2] += x0.z; acc[3] += x0.w; acc[4] += x1.x; acc[5] += x1.y; acc[6] += x1.z; acc[7] += x1.w;
            }
        };
        for (int s = 0; s < T; ++s) {
            const int t = d == 0 ? T - 1 - s : s;
            const bool first = d == 0 ? t == 0 : t == T - 1;
            float vr[8], vz[8], vn[8], vhn[8], vhp[8], vdy[8];
            {
                const int st = s % NSB;
                if (ok) ok = tc::mbar_wait(&in_full[st], (s / NSB) & 1, p.dbg, 0x4200 + (s & 0xff));
                const uint32_t gp = sIn_u + (uint32_t)st * BWD_STAGE + 16u * tid;
                const uint4 u0 = tc::lds_u4(gp), u1 = tc::lds_u4(gp + 4096), u2 = tc::lds_u4(gp + 8192), u3 = tc::lds_u4(gp + 12288);
                uint4 uh = make_uint4(0u, 0u, 0u, 0u);
                float4 y0 = make_float4(0.f, 0.f, 0.f, 0.f), y1 = y0;
                if (!first) uh = tc::lds_u4(gp + G_BLOCK);
                if (!top) { y0 = tc::lds_f4(sIn_u + (uint32_t)st * BWD_STAGE + G_BLOCK + YB_BLOCK + 32u * tid); y1 = tc::lds_f4(sIn_u + (uint32_t)st * BWD_STAGE + G_BLOCK + YB_BLOCK + 32u * tid + 16); }
                unpack8(u0, vr); unpack8(u1, vz); unpack8(u2, vn); unpack8(u3, vhn); unpack8(uh, vhp);
                if (first && p.h0) {                        // the caller's initial state, in fp32
#pragma unroll
                    for (int i = 0; i < 8; ++i) vhp[i] = p.h0[((int64_t)d * B + tile * NB + c0 + i) * H + unit];
                }
                vdy[0] = y0.x; vdy[1] = y0.y; vdy[2] = y0.z; vdy[3] = y0.w; vdy[4] = y1.x; vdy[5] = y1.y; vdy[6] = y1.z; vdy[7] = y1.w;
                if (top) {
#pragma unroll
                    for (int i = 0; i < 8; ++i) vdy[i] = h_avg[i] + (h_arg[i] == t ? h_max[i] : 0.f);
                }
            }
            float c_n[8], c_r[8], c_z[8], pre[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float r = vr[i], z = vz[i], n = vn[i];
                c_n[i] = (1.f - z) * (1.f - n * n);
                c_r[i] = vhn[i] * r * (1.f - r);
                c_z[i] = (vhp[i] - n) * z * (1.f - z);
                pre[i] = dhz[i] + vdy[i];
            }
            float acc[8];
            const int buf = s & 1;
            if (s > 0) reduce_partials(s, acc);
            else {
#pragma unroll
                for (int i = 0; i < 8; ++i) acc[i] = 0.f;
            }
            const uint32_t tileb = sD_u + (uint32_t)sub * SUBD + (uint32_t)buf * DT_BYTES;
            const uint32_t nbuf = sN_u + (uint32_t)sub * SUBN + (uint32_t)buf * HS_CHUNK;
            float dar[8], daz[8], dan[8], danr[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float dh = acc[i] + pre[i];
                dan[i] = dh * c_n[i];
                dar[i] = dan[i] * c_r[i];
                daz[i] = dh * c_z[i];
                danr[i] = dan[i] * vr[i];
                dhz[i] = dh * vz[i];
                tc::sts_bf16(tileb + e_off[i], __float2bfloat16(dar[i]));
                tc::sts_bf16(tileb + HS_CHUNK + e_off[i], __float2bfloat16(daz[i]));
                tc::sts_bf16(tileb + 2 * HS_CHUNK + e_off[i], __float2bfloat16(danr[i]));
            }
            tc::tcgen05_fence_before();
            tc::fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(&epi_done[sub]);
            // the ring slot is released only here: the published dgh depends on every value loaded from it (see tc_scan.cuh)
            if (lane == 0) tc::mbar_arrive(&in_empty[s % NSB]);
#pragma unroll
            for (int i = 0; i < 8; ++i) tc::sts_bf16(nbuf + e_off[i], __float2bfloat16(dan[i]));
            tc::fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(&st_done[sub]);
#pragma unroll
            for (int i = 0; i < 8; ++i) { sb_r += dar[i]; sb_z += daz[i]; sb_n += dan[i]; sb_nr += danr[i]; }
        }
        float* dbi = p.db_ih + (int64_t)d * p.dir_stride;
        float* dbh = p.db_hh + (int64_t)d * p.dir_stride;
        atomicAdd(dbi + unit, sb_r); atomicAdd(dbi + H + unit, sb_z); atomicAdd(dbi + 2 * H + unit, sb_n);
        atomicAdd(dbh + unit, sb_r); atomicAdd(dbh + H + unit, sb_z); atomicAdd(dbh + 2 * H + unit, sb_nr);
        if (p.dh0) {
            // gradient of the initial hidden state = z-carry of the last step + W_hh^T dgh of the last step (one more product)
            float acc[8];
            reduce_partials(T, acc);
#pragma unroll
            for (int i = 0; i < 8; ++i) p.dh0[((int64_t)d * B + tile * NB + c0 + i) * H + unit] = dhz[i] + acc[i];
        }
    }
    tc::tcgen05_fence_before();
    __syncthreads();
    tc::cluster_sync_all();
    if (warp == EPI_WARPS) tc::tmem_dealloc(tmem, 512);
}

static inline cudaError_t launch_bwd(const BwdParams& p_in, cudaStream_t st) {
    BwdParams p = p_in;
    if (p.H != 512 || p.B % NB != 0) return cudaErrorInvalidValue;
    // the ping-pong form (two 16-row sub-tiles) is the default; BIGRU_W_BWD=single selects the single-tile kernel
    static const bool single = [] { const char* e = getenv("BIGRU_W_BWD"); return e && e[0] == 's'; }();
    const bool pp = !single;
    {
        const uint32_t box[2] = {64u, (uint32_t)(pp ? tcx::NBS : NB)};
        const uint64_t d1[2] = {(uint64_t)p.D * 3 * p.H, (uint64_t)p.T * p.B};
        const uint64_t s1[1] = {(uint64_t)p.D * 3 * p.H * 2};
        const uint64_t d2[2] = {(uint64_t)p.D * p.H, (uint64_t)p.T * p.B};
        const uint64_t s2[1] = {(uint64_t)p.D * p.H * 2};
        if (make_tmap_bf16(&p.tmGI, p.dgi_row, 2, d1, s1, box) != 0 || make_tmap_bf16(&p.tmGN, p.dghn_row, 2, d2, s2, box) != 0)
            return cudaErrorInvalidValue;
    }
    const int CS = p.H / UNITS;
    const size_t smem = bwd_smem_bytes(p.H);
    void (*kern)(BwdParams) = pp ? gru_scanw_bwd2_kernel<512> : gru_scanw_bwd_kernel<512>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
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

// ---- weight images ------------------------------------------------------------------------------
// forward  fimg[((d*CS + c)*128 + lane)*ROW + col]:  lane < 64: col < H -> W_hr[64c+lane][col], col >= H -> W_hn[64c+lane][col-H]
//                                                    (first KC_T*64 columns of W_hn); lane >= 64: col < H -> W_hz[64c+lane-64][col], else 0
//          ftail[(((d*CS + c)*NTAIL + t)*128 + row)*64 + k]: row < 64 -> W_hn[64c+row][(KC_T + t)*64 + k], else 0
// backward bimg[((d*CS + c)*128 + i)*(NRB*192) + rb*192 + g*64 + jj] = W_hh[g*H + 64c + jj][128*rb + i]
template <int H>
__global__ void pack_wide_images_kernel(const float* __restrict__ w_hh, __nv_bfloat16* __restrict__ fimg, __nv_bfloat16* __restrict__ ftail,
                                        __nv_bfloat16* __restrict__ bimg) {
    using G = Geo<H>;
    constexpr int CS = G::CS, ROW = G::ROW_ELEMS, KC_T = G::KC_T, NTAIL = G::NTAIL, NRB = G::NRB;
    const int64_t nthr = (int64_t)gridDim.x * blockDim.x, t0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (int64_t i = t0; i < (int64_t)CS * 128 * ROW; i += nthr) {
        const int c = (int)(i / (128 * ROW)), lane = (int)((i / ROW) % 128), col = (int)(i % ROW);
        float w = 0.f;
        if (lane < 64) w = col < H ? w_hh[((int64_t)0 * H + 64 * c + lane) * H + col] : w_hh[((int64_t)2 * H + 64 * c + lane) * H + (col - H)];
        else if (col < H) w = w_hh[((int64_t)1 * H + 64 * c + lane - 64) * H + col];
        fimg[i] = __float2bfloat16(w);
    }
    for (int64_t i = t0; i < (int64_t)CS * NTAIL * 128 * 64; i += nthr) {
        const int k = (int)(i % 64), row = (int)((i / 64) % 128), tl = (int)((i / (64 * 128)) % NTAIL), c = (int)(i / ((int64_t)64 * 128 * NTAIL));
        ftail[i] = __float2bfloat16(row < 64 ? w_hh[((int64_t)2 * H + 64 * c + row) * H + (KC_T + tl) * 64 + k] : 0.f);
    }
    for (int64_t i = t0; i < (int64_t)CS * 128 * NRB * 192; i += nthr) {
        const int c = (int)(i / ((int64_t)128 * NRB * 192));
        const int64_t r = i % ((int64_t)128 * NRB * 192);
        const int lane_i = (int)(r / (NRB * 192)), col = (int)(r % (NRB * 192));
        const int rb = col / 192, kq = col % 192, g = kq / 64, jj = kq % 64;
        bimg[i] = __float2bfloat16(w_hh[((int64_t)g * H + 64 * c + jj) * H + 128 * rb + lane_i]);
    }
}

}  // namespace tcw
