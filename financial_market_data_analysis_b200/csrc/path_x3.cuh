// path_x3.cuh - BIGRU_PREC_BF16X3: the fp32-class tensor-core path (BASELINE.json configs[1]: "fp32 tolerance check").
// Every tensor-core operand is a (hi, lo) pair of bf16 values, x = hi + lo to 2^-17 relative; products are formed as
//   GEMMs (projection, dX, dW):  A_hi B_hi + A_hi B_lo + A_lo B_hi                       (tc_gemm.cuh, nsplit = 3)
//   recurrences:                 (W_hi + W_lo)(h_hi + h_lo), W resident in tensor memory   (tc_scan_x.cuh)
// with fp32 accumulation, fp32 gate math / state / stash / gradients.  Same structure and time-major layouts as
// path_bf16.cuh; the blocked scan layouts are those of tc_scan_x.cuh (64 units per CTA, 32-row batch tiles).
// Supported: H in {128, 256}, B % 32 == 0, F % 8 == 0; an initial hidden state (biGRU_model.py:63 `hidden`) is supported.
#pragma once
#include "path_bf16.cuh"
#include "tc_scan_x.cuh"
#include <cstdlib>

static int x3_plan_check(const bigru_plan& p) {
    if ((p.H != 128 && p.H != 256) || p.B % 32 != 0) {
        bigru_set_error("BIGRU_PREC_BF16X3 supports hidden_size 128 or 256 and batch %% 32 == 0 (got H=%d B=%d; the Python mirror pads "
                        "other batch sizes with zero rows); use BIGRU_PREC_FP32 for other shapes", p.H, p.B);
        return BIGRU_ERR_UNSUPPORTED;
    }
    return BIGRU_OK;
}

struct X3Layout {              // byte offsets, 1024-aligned
    size_t Yhi[16], Ylo[16], YB[16], G[16], Xhi[16], Xlo[16];
    size_t Wih_hi[16], Wih_lo[16], WihT_hi[16], WihT_lo[16], Wimg[16], WTimg[16], bfold[16], bhn[16];
    size_t cat, arg, dbg, stash_total;
    size_t gi, dghn_hi, dghn_lo, dYa, dYb, gh0, scratch_total;
};
static X3Layout x3_layout(const bigru_plan& p) {
    X3Layout L{};
    const size_t R = (size_t)p.B * p.T, DH = (size_t)p.D * p.H, H = p.H, D = p.D;
    size_t o = 0;
    for (int l = 0; l < p.L; ++l) {
        const size_t I = p.in_size(l), Ip = (size_t)pad8((int64_t)I);      // layer-0 K extent padded to 8 (see path_bf16.cuh)
        L.Yhi[l] = o; o = al(o + R * DH * 2);
        L.Ylo[l] = o; o = al(o + R * DH * 2);
        L.YB[l] = o; o = al(o + R * DH * 4);
        L.G[l] = o; o = al(o + R * D * 4 * H * 4);
        L.Xhi[l] = o; o = al(o + R * Ip * 2);
        L.Xlo[l] = o; o = al(o + R * Ip * 2);
        L.Wih_hi[l] = o; o = al(o + D * 3 * H * Ip * 2);
        L.Wih_lo[l] = o; o = al(o + D * 3 * H * Ip * 2);
        L.WihT_hi[l] = o; o = al(o + D * 3 * H * I * 2);
        L.WihT_lo[l] = o; o = al(o + D * 3 * H * I * 2);
        L.Wimg[l] = o; o = al(o + D * 2 * 3 * H * H * 2);        // stacked hi | lo rows
        L.WTimg[l] = o; o = al(o + D * 2 * 3 * H * H * 2);
        L.bfold[l] = o; o = al(o + D * 3 * H * 4);
        L.bhn[l] = o; o = al(o + D * H * 4);
    }
    L.cat = o; o = al(o + (size_t)p.B * 3 * H * 4);
    L.arg = o; o = al(o + (size_t)p.B * H * 4);
    L.dbg = o; o = al(o + 256);
    L.stash_total = o;
    o = 0;
    const size_t wide = DH > (size_t)p.F ? DH : (size_t)p.F;
    L.gi = o; o = al(o + R * D * 3 * H * 4);                     // forward: giX fp32; backward: dgi_hi | dgi_lo (bf16 each)
    L.dghn_hi = o; o = al(o + R * D * H * 2);
    L.dghn_lo = o; o = al(o + R * D * H * 2);
    L.dYa = o; o = al(o + R * wide * 4);
    L.dYb = o; o = al(o + R * wide * 4);
    L.gh0 = o; o = al(o + (size_t)p.B * D * 3 * H * 4);          // W_hh h0 of the layer being scanned (initial state given)
    L.scratch_total = o;
    return L;
}
static void x3_workspace(const bigru_plan& p, size_t* a, size_t* b) {
    const X3Layout L = x3_layout(p);
    *a = L.stash_total; *b = L.scratch_total;
}

// ---------------------------------------------------------------------------------------------------
// small kernels of this path
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void x3_split(float x, bf16_t& hi, bf16_t& lo) {
    hi = __float2bfloat16(x);
    lo = __float2bfloat16(x - __bfloat162float(hi));
}

// inter-layer dropout on the split layer output: (hi + lo) masked and re-split
__global__ void x3_dropout_rows_kernel(const bf16_t* __restrict__ Yhi, const bf16_t* __restrict__ Ylo, bf16_t* __restrict__ Xhi,
                                       bf16_t* __restrict__ Xlo, int64_t R, int cols, int B, int T, float pdrop, uint64_t seed, uint32_t stream) {
    const float scale = 1.f / (1.f - pdrop);
    const int64_t total = R * cols;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int cidx = i % cols;
        const int64_t r = i / cols;
        const int64_t b = r % B, t = r / B;
        const uint64_t key = ((uint64_t)b * T + t) * cols + cidx;
        const float v = bigru_uniform(seed, stream, key) < pdrop ? 0.f : (__bfloat162float(Yhi[i]) + __bfloat162float(Ylo[i])) * scale;
        bf16_t hi, lo;
        x3_split(v, hi, lo);
        Xhi[i] = hi; Xlo[i] = lo;
    }
}
// gradient of the same dropout, in place on the blocked fp32 gradient of tc_scan_x.cuh: [d][tile][t][cta][thread][8]
__global__ void x3_dropout_grad_rows_kernel(float* __restrict__ dYB, int64_t R, int cols, int B, int T, int H, float pdrop,
                                            uint64_t seed, uint32_t stream) {
    const float scale = 1.f / (1.f - pdrop);
    const int64_t total = R * cols;
    const int CS = H / 64, ntl = B / 32;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int i8 = i & 7;
        int64_t e = i >> 3;
        const int tid = e % 256; e /= 256;
        const int c = e % CS; e /= CS;
        const int t = e % T; e /= T;
        const int tile = e % ntl;
        const int d = e / ntl;
        const int unit = c * 64 + (tid & 63);
        const int64_t b = tile * 32 + (tid >> 6) * 8 + i8;
        const uint64_t key = ((uint64_t)b * T + t) * cols + (uint64_t)(d * H + unit);
        dYB[i] = bigru_uniform(seed, stream, key) < pdrop ? 0.f : dYB[i] * scale;
    }
}

// All weight packing of a forward call in one launch: blockIdx.y enumerates (layer, direction).
struct X3PackJob { const float* w_ih; const float* w_hh; const float* b_ih; const float* b_hh;
                   bf16_t *Wih_hi, *Wih_lo, *WihT_hi, *WihT_lo, *Wimg, *WTimg; float* bfold; float* bhn; int I; int d; };
struct X3PackJobs { X3PackJob j[32]; };
__global__ void __launch_bounds__(256) x3_pack_all_kernel(const X3PackJobs jobs, int H, int D) {
    __shared__ float tile[32][33];
    const X3PackJob& J = jobs.j[blockIdx.y];
    const int H3 = 3 * H, I = J.I, d = J.d;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    // W_ih [3H][I] -> rows d*3H.. of Wih_{hi,lo} [D*3H][I] and columns d*3H.. of WihT_{hi,lo} [I][D*3H]
    if (I % 32 == 0) {
        const int tr = H3 / 32, tcn = I / 32;
        for (int tl = blockIdx.x; tl < tr * tcn; tl += gridDim.x) {
            const int r0 = (tl / tcn) * 32, c0 = (tl % tcn) * 32;
#pragma unroll
            for (int i = ty; i < 32; i += 8) {
                const float v = J.w_ih[(int64_t)(r0 + i) * I + c0 + tx];
                tile[i][tx] = v;
                bf16_t hi, lo;
                x3_split(v, hi, lo);
                const int64_t o = ((int64_t)d * H3 + r0 + i) * I + c0 + tx;
                J.Wih_hi[o] = hi; J.Wih_lo[o] = lo;
            }
            __syncthreads();
#pragma unroll
            for (int i = ty; i < 32; i += 8) {
                bf16_t hi, lo;
                x3_split(tile[tx][i], hi, lo);
                const int64_t o = (int64_t)(c0 + i) * D * H3 + (int64_t)d * H3 + r0 + tx;
                J.WihT_hi[o] = hi; J.WihT_lo[o] = lo;
            }
            __syncthreads();
        }
    } else {
        const int Ip = (I + 7) & ~7;                           // zero columns up to the padded row pitch
        const int64_t n_ih = (int64_t)H3 * Ip;
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_ih; i += (int64_t)gridDim.x * blockDim.x) {
            const int k = i % Ip, q = i / Ip;
            bf16_t hi, lo;
            x3_split(k < I ? J.w_ih[(int64_t)q * I + k] : 0.f, hi, lo);
            const int64_t o1 = ((int64_t)d * H3 + q) * Ip + k, o2 = (int64_t)k * D * H3 + (int64_t)d * H3 + q;
            J.Wih_hi[o1] = hi; J.Wih_lo[o1] = lo;
            if (k < I) { J.WihT_hi[o2] = hi; J.WihT_lo[o2] = lo; }
        }
    }
    // W_hh -> the forward (stacked hi | lo rows) and backward (own-gate rows x all k) tensor-memory images of tc_scan_x.cuh
    {
        const int CS = H / 64, NKH = H / 128, NRB = 2 * NKH;
        const int64_t per_cta = (int64_t)128 * 3 * H;
        const int64_t total = (int64_t)CS * per_cta;
        bf16_t* fimg = J.Wimg + (int64_t)d * total;
        bf16_t* bimg = J.WTimg + (int64_t)d * total;
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
            const int c = (int)(i / per_cta);
            const int64_t r = i % per_cta;
            {
                const int row = (int)(r / (3 * H)), col = (int)(r % (3 * H));
                const int g = col / H, k = col % H, part = row >> 6, jj = row & 63;
                bf16_t hi, lo;
                x3_split(J.w_hh[((int64_t)g * H + 64 * c + jj) * H + k], hi, lo);
                fimg[i] = part ? lo : hi;
            }
            {
                const int lane_i = (int)(r / (NRB * 192)), col = (int)(r % (NRB * 192));
                const int rb = col / 192, kq = col % 192, g = kq / 64, jj = kq % 64;
                const int part = rb / NKH, kh = rb % NKH;
                bf16_t hi, lo;
                x3_split(J.w_hh[((int64_t)g * H + 64 * c + jj) * H + 128 * kh + lane_i], hi, lo);
                bimg[i] = part ? lo : hi;
            }
        }
    }
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < H3; q += (int64_t)gridDim.x * blockDim.x) {
        J.bfold[d * H3 + q] = J.b_ih[q] + (q < 2 * H ? J.b_hh[q] : 0.f);
        if (q >= 2 * H) J.bhn[d * H + q - 2 * H] = J.b_hh[q];
    }
}

// ---------------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------------
static int forward_x3(const bigru_plan& p, const float* params, const float* x, const float* h0, float drop,
                      int spatial, int training, uint64_t seed, void* stash_v, void* scratch_v, float* logits,
                      float* hn, cudaStream_t st, WindowSrc win = WindowSrc{nullptr, nullptr, nullptr, 0}) {
    const X3Layout L = x3_layout(p);
    uint8_t* S = (uint8_t*)stash_v;
    uint8_t* W = (uint8_t*)scratch_v;
    const int B = p.B, T = p.T, H = p.H, D = p.D, F = p.F;
    const int64_t R = (int64_t)B * T;
    const bool do_drop = training && drop > 0.f;
    unsigned int* dbg = (unsigned int*)(S + L.dbg);
    CUDA_TRY(cudaMemsetAsync(dbg, 0, 64, st));
    {
        X3PackJobs jobs{};
        int nj = 0;
        for (int l = 0; l < p.L; ++l)
            for (int d = 0; d < D; ++d) {
                X3PackJob& J = jobs.j[nj++];
                J.w_ih = params + p.off_wih(l, d); J.w_hh = params + p.off_whh(l, d);
                J.b_ih = params + p.off_bih(l, d); J.b_hh = params + p.off_bhh(l, d);
                J.Wih_hi = (bf16_t*)(S + L.Wih_hi[l]); J.Wih_lo = (bf16_t*)(S + L.Wih_lo[l]);
                J.WihT_hi = (bf16_t*)(S + L.WihT_hi[l]); J.WihT_lo = (bf16_t*)(S + L.WihT_lo[l]);
                J.Wimg = (bf16_t*)(S + L.Wimg[l]); J.WTimg = (bf16_t*)(S + L.WTimg[l]);
                J.bfold = (float*)(S + L.bfold[l]); J.bhn = (float*)(S + L.bhn[l]); J.I = (int)p.in_size(l); J.d = d;
            }
        KLAUNCH(KC_PACK, 0.0, 0.0, st, x3_pack_all_kernel<<<dim3(148, nj), 256, 0, st>>>(jobs, H, D));
    }
    const bool direct = windows_direct(p, win.src != nullptr, do_drop);      // zero-copy windows: only the chunk is normalised and split
    if (direct)
        KLAUNCH(KC_PACK, 0.0, 8.0 * (B + T - 1) * F, st, chunk_prep_kernel<<<148, 256, 0, st>>>(win, (bf16_t*)(S + L.Xhi[0]), (bf16_t*)(S + L.Xlo[0]),
                                                                                                 (int64_t)B + T - 1, F));
    else if (F % 8 == 0)
        KLAUNCH(KC_PACK, 0.0, 8.0 * R * F, st, cast_x_kernel<<<148 * 8, 256, 0, st>>>(x, win, (bf16_t*)(S + L.Xhi[0]), (bf16_t*)(S + L.Xlo[0]), B, T, F,
                                                                                       do_drop ? drop : 0.f, spatial, seed));
    else
        KLAUNCH(KC_PACK, 0.0, 8.0 * R * F, st, cast_x_pad_kernel<<<148 * 8, 256, 0, st>>>(x, win, (bf16_t*)(S + L.Xhi[0]), (bf16_t*)(S + L.Xlo[0]), B, T, F,
                                                                                           pad8(F), do_drop ? drop : 0.f, spatial, seed));
    for (int l = 0; l < p.L; ++l) {
        const int I = (int)p.in_size(l);
        const bf16_t* Xhi = (const bf16_t*)(S + L.Xhi[l]);
        const bf16_t* Xlo = (const bf16_t*)(S + L.Xlo[l]);
        if (l > 0) {
            if (do_drop) {
                KLAUNCH(KC_MISC, 0.0, 0.0, st, x3_dropout_rows_kernel<<<148 * 8, 256, 0, st>>>(
                                                   (const bf16_t*)(S + L.Yhi[l - 1]), (const bf16_t*)(S + L.Ylo[l - 1]), (bf16_t*)(S + L.Xhi[l]),
                                                   (bf16_t*)(S + L.Xlo[l]), R, I, B, T, drop, seed, (uint32_t)l));
            } else {
                Xhi = (const bf16_t*)(S + L.Yhi[l - 1]); Xlo = (const bf16_t*)(S + L.Ylo[l - 1]);
            }
        }
        {   // input projection for all t, both directions: W_ih X^T + bias(row) in the scan kernel's blocked fp32 layout
            tcg::Params g{};
            const int Ip = pad8(I);                                                     // zero-padded K extent (layer 0, n_features % 8 != 0)
            g.M = D * 3 * H; g.N = (int)R; g.K = Ip; g.batch = 1; g.splitk = 1; g.mode = tcg::OUT_SCAN_F32;
            g.blk = tcg::ScanBlk{T, B, H, 3, 64, 32}; g.m_fast = 1;
            g.C = W + L.gi; g.ldc = R; g.bias = (const float*)(S + L.bfold[l]); g.bias_per_row = 1; g.dbg = dbg;
            const bool wnd = direct && l == 0;
            g.b_win = wnd ? B : 0;
            TRY(tc_gemm(S + L.Wih_hi[l], D * 3 * H, Ip, Xhi, wnd ? (int64_t)B + T - 1 : R, Ip, g, st, KC_TC_GEMM, S + L.Wih_lo[l], Xlo));
        }
        if (h0) {   // recurrent product of the initial state, exact fp32 (tiny: B x 3H x H per direction); the scan starts at step 1
            GemmArgs r = gemm_args(h0 + (int64_t)l * D * B * H, params + p.off_whh(l, 0), (float*)(W + L.gh0), B, 3 * H, H, H, 1, H, 1, 3 * H);
            r.batch = D; r.zA = (int64_t)B * H; r.zB = p.ld_block(l); r.zC = (int64_t)B * 3 * H;
            TRY(sgemm_launch(r, st));
        }
        tcx::FwdParams f{};
        f.B = B; f.T = T; f.H = H; f.D = D;
        f.Wimg = (const bf16_t*)(S + L.Wimg[l]); f.giX = (const float*)(W + L.gi); f.b_hn = (const float*)(S + L.bhn[l]);
        f.h0 = h0 ? h0 + (int64_t)l * D * B * H : nullptr;
        f.gh0 = h0 ? (const float*)(W + L.gh0) : nullptr;
        f.GX = (float*)(S + L.G[l]); f.YBX = (float*)(S + L.YB[l]);
        f.hn_out = hn ? hn + (int64_t)l * D * B * H : nullptr;
        f.Yhi = (bf16_t*)(S + L.Yhi[l]); f.Ylo = (bf16_t*)(S + L.Ylo[l]); f.dbg = dbg;
        {
            ProfScope ps(KC_TC_SCAN_FWD, 2.0 * 3 * H * H * (double)R * D, 0.0, st);
            CUDA_TRY(tcx::launch_fwd(f, st));
        }
    }
    {
        const int G = 256 / (H / 8);
        const size_t hsm = sizeof(float) * ((size_t)3 * G * H + (size_t)p.C * 8);
        KLAUNCH(KC_HEAD, 0.0, 4.0 * R * D * H, st, head_fwd_kernel<<<B, 256, hsm, st>>>(
                    (const bf16_t*)(S + L.Yhi[p.L - 1]), (const bf16_t*)(S + L.Ylo[p.L - 1]), params + p.off_linw(), params + p.off_linb(),
                    (float*)(S + L.cat), (int*)(S + L.arg), logits, B, T, H, D, p.C));
    }
    return BIGRU_OK;
}

// ---------------------------------------------------------------------------------------------------
// backward
// ---------------------------------------------------------------------------------------------------
static int backward_x3(const bigru_plan& p, const float* params, const float* x, const float* h0, float drop,
                       int spatial, int training, uint64_t seed, const void* stash_v, void* scratch_v,
                       const float* dlogits, float* grads, float* dx, float* dh0, cudaStream_t st, int l_from = -1, int l_to = 0) {
    // layers l_from .. l_to (downwards; l_from = -1: from the top layer).  A call that starts at the top layer also zeroes the gradient
    // vector and forms the head's gradients; a later call for the lower layers continues from the dY the upper call left in scratch.
    if (l_from < 0) l_from = p.L - 1;
    const bool from_top = l_from == p.L - 1;
    const X3Layout L = x3_layout(p);
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
    bf16_t* dgi_hi = (bf16_t*)(W + L.gi);
    bf16_t* dgi_lo = dgi_hi + (size_t)R * D * 3 * H;
    bf16_t* dghn_hi = (bf16_t*)(W + L.dghn_hi);
    bf16_t* dghn_lo = (bf16_t*)(W + L.dghn_lo);
    for (int l = l_from; l >= l_to; --l) {
        const int I = (int)p.in_size(l);
        tcx::BwdParams b{};
        b.B = B; b.T = T; b.H = H; b.D = D;
        b.WTimg = (const bf16_t*)(S + L.WTimg[l]); b.GX = (const float*)(S + L.G[l]); b.YBX = (const float*)(S + L.YB[l]);
        b.dYBX = dY;
        b.h0 = h0 ? h0 + (int64_t)l * D * B * H : nullptr;
        b.dh0 = dh0 ? dh0 + (int64_t)l * D * B * H : nullptr;
        if (l == p.L - 1) { b.dlogits = dlogits; b.lin_w = params + p.off_linw(); b.arg = (const int*)(S + L.arg); b.C = C; }
        b.dgi_hi = dgi_hi; b.dgi_lo = dgi_lo; b.dghn_hi = dghn_hi; b.dghn_lo = dghn_lo;
        b.db_ih = grads + p.off_bih(l, 0); b.db_hh = grads + p.off_bhh(l, 0); b.dir_stride = p.ld_block(l); b.dbg = dbg;
        {
            ProfScope ps(KC_TC_SCAN_BWD, 2.0 * 3 * H * H * (double)R * D, 0.0, st);
            CUDA_TRY(tcx::launch_bwd(b, st));
        }
        const bool dropped = do_drop && (l == 0 || p.L > 1);
        const bool own_x = l == 0 || dropped;
        const bf16_t* Xin_hi = own_x ? (const bf16_t*)(S + L.Xhi[l]) : (const bf16_t*)(S + L.Yhi[l - 1]);
        const bf16_t* Xin_lo = own_x ? (const bf16_t*)(S + L.Xlo[l]) : (const bf16_t*)(S + L.Ylo[l - 1]);
        {   // dW_ih[d] = dgi[d]^T X
            tcg::Params g{};
            g.M = 3 * H; g.N = I; g.K = (int)R; g.batch = D; g.mode = tcg::OUT_ATOMIC_F32; g.a_mn = 1; g.b_mn = 1;
            const int tiles = ((3 * H + 127) / 128) * ((I + 127) / 128) * D;
            g.splitk = (int)std::max<int64_t>(1, std::min<int64_t>((R + 63) / 64, (148 * 2 + tiles / 2) / tiles));
            g.C = grads + p.off_wih(l, 0); g.ldc = I; g.zC = p.ld_block(l);
            for (int d = 0; d < D; ++d) { g.a_row_off[d] = d * 3 * H; g.b_row_off[d] = 0; g.b_k_off[d] = 0; }
            g.dbg = dbg;
            g.b_win = (l == 0 && windows_direct(p, x == nullptr, do_drop)) ? B : 0;      // forward_windows left only the chunk in the stash
            g.b_win_rows = B + T - 1;
            TRY(tc_gemm(dgi_hi, (int64_t)D * 3 * H, (int64_t)D * 3 * H, Xin_hi, I, pad8(I), g, st, KC_TC_GEMM_DWIH, dgi_lo, Xin_lo));   // I columns, padded pitch
        }
        for (int part = 0; part < 2; ++part) {   // dW_hh[d] = dgh[d]^T H_prev (time-shifted Y, see path_bf16.cuh)
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
            if (part == 0) TRY(tc_gemm(dgi_hi, (int64_t)D * 3 * H, (int64_t)D * 3 * H, S + L.Yhi[l], (int64_t)D * H, (int64_t)D * H, g, st, KC_TC_GEMM_DWHH, dgi_lo, S + L.Ylo[l]));
            else TRY(tc_gemm(dghn_hi, (int64_t)D * H, (int64_t)D * H, S + L.Yhi[l], (int64_t)D * H, (int64_t)D * H, g, st, KC_TC_GEMM_DWHH, dghn_lo, S + L.Ylo[l]));
        }
        if (h0)   // the first step's h_prev term of dW_hh (dwhh_h0_kernel, path_bf16.cuh)
            KLAUNCH(KC_MISC, 0.0, 0.0, st, dwhh_h0_kernel<<<dim3((3 * H + 127) / 128, H / DWHH_H0_COLS, D), 128, 0, st>>>(
                        dgi_hi, dgi_lo, dghn_hi, dghn_lo, h0 + (int64_t)l * D * B * H, grads + p.off_whh(l, 0), p.ld_block(l), B, T, H, D));
        const bool need_dx = l > 0 || dx != nullptr;
        if (need_dx) {   // dX^T = W_ih^T (both directions along K = D*3H) x dgi^T
            tcg::Params g{};
            g.M = I; g.N = (int)R; g.K = D * 3 * H; g.batch = 1; g.splitk = 1;
            g.mode = l > 0 ? tcg::OUT_SCAN_F32 : tcg::OUT_F32;
            g.blk = tcg::ScanBlk{T, B, H, 1, 64, 32}; g.m_fast = 1;
            g.C = dYnext; g.ldc = R; g.dbg = dbg;
            TRY(tc_gemm(S + L.WihT_hi[l], I, (int64_t)D * 3 * H, dgi_hi, R, (int64_t)D * 3 * H, g, st, KC_TC_GEMM_DX, S + L.WihT_lo[l], dgi_lo));
            if (l > 0 && dropped)
                KLAUNCH(KC_MISC, 0.0, 0.0, st, x3_dropout_grad_rows_kernel<<<148 * 8, 256, 0, st>>>(dYnext, R, I, B, T, H, drop, seed, (uint32_t)l));
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
