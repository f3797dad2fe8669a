// api.cu - extern "C" entry points of libbigru_b200.so (see include/bigru_b200.h).
#include "common.cuh"
#include "kernels_f32.cuh"
#include "path_bf16.cuh"
#include "path_x3.cuh"
#include "features.cuh"
#include "infer_small.cuh"
#include "infer_cluster.cuh"

#include <cstdlib>
#include <cstring>
#include <new>

static thread_local char g_err[512] = "";
void bigru_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

extern "C" const char* bigru_last_error(void) { return g_err; }
extern "C" int bigru_version(void) { return 200; }

extern "C" int bigru_device_check(int dev) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || dev >= n) {
        cudaGetLastError();
        bigru_set_error("no CUDA device %d (libbigru_b200 has no CPU fallback)", dev);
        return BIGRU_ERR_DEVICE;
    }
    cudaDeviceProp p;
    CUDA_TRY(cudaGetDeviceProperties(&p, dev));
    if (p.major != 10) {
        bigru_set_error("device %d is sm_%d%d; libbigru_b200 is built for sm_100a only", dev, p.major, p.minor);
        return BIGRU_ERR_DEVICE;
    }
    return BIGRU_OK;
}

// ------------------------------------------------------------------------------------------
// workspace carve-up (fp32 path).  Offsets in floats.
// ------------------------------------------------------------------------------------------
struct StashF32 {       // kept forward -> backward
    int64_t Y[16], G[16], X[16];   // per layer: output [B*T*D*H], gates [D][B*T][4H], dropped input [B*T*I_l]
    int64_t cat, arg, total;
};
struct ScratchF32 {
    int64_t gi, gh, dgi, dgh, dYa, dYb, dhc, dcat, total;
};
static StashF32 stash_layout(const bigru_plan& p) {
    StashF32 s{};
    int64_t o = 0;
    const int64_t BT = (int64_t)p.B * p.T;
    for (int l = 0; l < p.L; ++l) {
        s.Y[l] = o; o += BT * p.D * p.H;
        s.G[l] = o; o += (int64_t)p.D * BT * 4 * p.H;
        s.X[l] = o; o += BT * p.in_size(l);
    }
    s.cat = o; o += (int64_t)p.B * 3 * p.H;
    s.arg = o; o += (int64_t)p.B * p.H;
    s.total = o;
    return s;
}
static ScratchF32 scratch_layout(const bigru_plan& p) {
    ScratchF32 s{};
    int64_t o = 0;
    const int64_t BT = (int64_t)p.B * p.T;
    const int64_t wide = p.D * p.H > p.F ? p.D * p.H : p.F;
    s.gi = o; o += (int64_t)p.D * BT * 3 * p.H;
    s.gh = o; o += (int64_t)p.D * p.B * 3 * p.H;
    s.dgi = o; o += (int64_t)p.D * BT * 3 * p.H;
    s.dgh = o; o += (int64_t)p.D * BT * 3 * p.H;
    s.dYa = o; o += BT * wide;
    s.dYb = o; o += BT * wide;
    s.dhc = o; o += (int64_t)p.D * p.B * p.H;
    s.dcat = o; o += (int64_t)p.B * 3 * p.H;
    s.total = o;
    return s;
}

extern "C" int bigru_plan_create(int B, int T, int F, int H, int L, int C, int bidirectional, int precision,
                                 bigru_plan** out) {
    if (!out) { bigru_set_error("plan_create: out is null"); return BIGRU_ERR_ARG; }
    if (B <= 0 || T <= 0 || F <= 0 || H <= 0 || L <= 0 || L > 16 || C <= 0) {
        bigru_set_error("plan_create: bad shape B=%d T=%d F=%d H=%d L=%d C=%d", B, T, F, H, L, C);
        return BIGRU_ERR_ARG;
    }
    if (precision != BIGRU_PREC_FP32 && precision != BIGRU_PREC_BF16 && precision != BIGRU_PREC_BF16X3) {
        bigru_set_error("plan_create: unknown precision %d", precision);
        return BIGRU_ERR_ARG;
    }
    bigru_plan* p = new (std::nothrow) bigru_plan();
    if (!p) { bigru_set_error("plan_create: out of host memory"); return BIGRU_ERR_ARG; }
    p->B = B; p->T = T; p->F = F; p->H = H; p->L = L; p->C = C; p->D = bidirectional ? 2 : 1; p->prec = precision;
    p->nparams = p->off_linb() + C;
    if (precision == BIGRU_PREC_BF16) {
        int rc = bf16_plan_check(*p);
        if (rc != BIGRU_OK) { delete p; return rc; }
        bf16_workspace(*p, &p->stash_bytes, &p->scratch_bytes);
    } else if (precision == BIGRU_PREC_BF16X3) {
        int rc = x3_plan_check(*p);
        if (rc != BIGRU_OK) { delete p; return rc; }
        x3_workspace(*p, &p->stash_bytes, &p->scratch_bytes);
    } else {
        p->stash_bytes = (size_t)stash_layout(*p).total * sizeof(float);
        p->scratch_bytes = (size_t)scratch_layout(*p).total * sizeof(float);
    }
    *out = p;
    return BIGRU_OK;
}

extern "C" int bigru_plan_destroy(bigru_plan* plan) { delete plan; return BIGRU_OK; }
extern "C" int64_t bigru_param_count(const bigru_plan* plan) { return plan ? plan->nparams : -1; }

extern "C" int bigru_param_offset(const bigru_plan* p, int layer, int dir, int which, int64_t* offset,
                                  int64_t* rows, int64_t* cols) {
    if (!p || !offset || !rows || !cols || layer < 0 || layer > p->L || dir < 0 || dir >= p->D || which < 0 || which > 3) {
        bigru_set_error("param_offset: bad argument");
        return BIGRU_ERR_ARG;
    }
    if (layer == p->L) {
        if (which == 0) { *offset = p->off_linw(); *rows = p->C; *cols = 3 * p->H; }
        else if (which == 2) { *offset = p->off_linb(); *rows = p->C; *cols = 1; }
        else { bigru_set_error("param_offset: linear has which 0 (weight) or 2 (bias)"); return BIGRU_ERR_ARG; }
        return BIGRU_OK;
    }
    switch (which) {
        case 0: *offset = p->off_wih(layer, dir); *rows = 3 * p->H; *cols = p->in_size(layer); break;
        case 1: *offset = p->off_whh(layer, dir); *rows = 3 * p->H; *cols = p->H; break;
        case 2: *offset = p->off_bih(layer, dir); *rows = 3 * p->H; *cols = 1; break;
        default: *offset = p->off_bhh(layer, dir); *rows = 3 * p->H; *cols = 1; break;
    }
    return BIGRU_OK;
}

extern "C" int bigru_workspace_bytes(const bigru_plan* p, size_t* stash_bytes, size_t* scratch_bytes) {
    if (!p || !stash_bytes || !scratch_bytes) { bigru_set_error("workspace_bytes: null argument"); return BIGRU_ERR_ARG; }
    *stash_bytes = p->stash_bytes;
    *scratch_bytes = p->scratch_bytes;
    return BIGRU_OK;
}

// where the head keeps argmax_t of the pooled output (int32 [B][H]) inside the stash of the last forward
extern "C" int bigru_stash_argmax_offset(const bigru_plan* p, size_t* byte_offset) {
    if (!p || !byte_offset) { bigru_set_error("stash_argmax_offset: null argument"); return BIGRU_ERR_ARG; }
    if (p->prec == BIGRU_PREC_BF16) *byte_offset = bf16_layout(*p).arg;
    else if (p->prec == BIGRU_PREC_BF16X3) *byte_offset = x3_layout(*p).arg;
    else *byte_offset = (size_t)stash_layout(*p).arg * sizeof(float);
    return BIGRU_OK;
}

static inline unsigned nblk(int64_t n, int bs) { return (unsigned)cdiv64(n, bs); }

// ------------------------------------------------------------------------------------------
// fp32 forward
// ------------------------------------------------------------------------------------------
static int forward_f32(const bigru_plan& p, const float* params, const float* x, const float* h0, float drop,
                       int spatial, int training, uint64_t seed, float* stash, float* scratch, float* logits,
                       float* hn, cudaStream_t st) {
    const StashF32 S = stash_layout(p);
    const ScratchF32 W = scratch_layout(p);
    const int B = p.B, T = p.T, H = p.H, D = p.D;
    const int64_t BT = (int64_t)B * T;
    const bool do_drop = training && drop > 0.f;
    const float* inp = x;
    for (int l = 0; l < p.L; ++l) {
        const int I = (int)p.in_size(l);
        if (do_drop && (l == 0 || p.L > 1)) {
            // l == 0: input dropout (elementwise or per-channel); l > 0: nn.GRU inter-layer dropout
            float* xd = stash + S.X[l];
            KLAUNCH(KC_MISC, 0.0, 0.0, st, dropout_kernel<<<148 * 8, 256, 0, st>>>(inp, xd, BT * I, T, I, l == 0 ? spatial : 0, drop, seed, (uint32_t)l));
            inp = xd;
        }
        // gi[d] = X W_ih[d]^T + b_ih[d]   for both directions
        GemmArgs g = gemm_args(inp, params + p.off_wih(l, 0), scratch + W.gi, (int)BT, 3 * H, I, I, 1, I, 1, 3 * H);
        g.bias = params + p.off_bih(l, 0);
        g.batch = D; g.zA = 0; g.zB = p.ld_block(l); g.zBias = p.ld_block(l); g.zC = BT * 3 * H;
        TRY(sgemm_launch(g, st));
        float* Y = stash + S.Y[l];
        float* G = stash + S.G[l];
        const float* h0l = h0 ? h0 + (int64_t)l * D * B * H : nullptr;
        float* hnl = hn ? hn + (int64_t)l * D * B * H : nullptr;
        for (int s = 0; s < T; ++s) {
            // gh[d] = h_prev[d] W_hh[d]^T + b_hh[d];  h_prev rows live in Y (or h0 at s == 0)
            const float* hp; int64_t sam, zA;
            if (s == 0) { hp = h0l; sam = H; zA = (int64_t)B * H; }
            else {
                // direction 0 reads t = s-1, direction 1 reads t = T-s; express via base pointer + batch stride
                hp = Y + (int64_t)(s - 1) * D * H;
                sam = (int64_t)T * D * H;
                zA = D == 2 ? ((int64_t)(T - s) - (s - 1)) * D * H + H : 0;
            }
            GemmArgs r = gemm_args(hp, params + p.off_whh(l, 0), scratch + W.gh, B, 3 * H, hp ? H : 0, sam, 1, H, 1, 3 * H);
            r.bias = params + p.off_bhh(l, 0);
            r.batch = D; r.zA = zA; r.zB = p.ld_block(l); r.zBias = p.ld_block(l); r.zC = (int64_t)B * 3 * H;
            if (hp) { TRY(sgemm_launch(r, st)); }
            else {
                // zero initial state: gh = b_hh
                r.A = params; r.K = 1; r.sam = 0; r.sak = 1; r.zA = 0;       // dummy operand, masked out below
                r.mask_period = 1; r.mask_skip = 0;                           // every k masked -> pure bias
                TRY(sgemm_launch(r, st));
            }
            KLAUNCH(KC_GATES_FWD, 0.0, 0.0, st, gru_gates_fwd_kernel<<<nblk((int64_t)D * B * H, 256), 256, 0, st>>>(scratch + W.gi, scratch + W.gh, h0l, Y, G,
                                                                              hnl, B, T, H, D, s));
        }
        inp = Y;
    }
    const float* Ytop = stash + S.Y[p.L - 1];
    KLAUNCH(KC_HEAD, 0.0, 0.0, st, head_pool_kernel<<<nblk((int64_t)B * H, 128), 128, 0, st>>>(Ytop, stash + S.cat, (int*)(stash + S.arg), B, T, H, D));
    GemmArgs lin = gemm_args(stash + S.cat, params + p.off_linw(), logits, B, p.C, 3 * H, 3 * H, 1, 3 * H, 1, p.C);
    lin.bias = params + p.off_linb();
    TRY(sgemm_launch(lin, st));
    return BIGRU_OK;
}

// ------------------------------------------------------------------------------------------
// fp32 backward
// ------------------------------------------------------------------------------------------
static int backward_f32(const bigru_plan& p, const float* params, const float* x, const float* h0, float drop,
                        int spatial, int training, uint64_t seed, const float* stash, float* scratch,
                        const float* dlogits, float* grads, float* dx, float* dh0, cudaStream_t st) {
    const StashF32 S = stash_layout(p);
    const ScratchF32 W = scratch_layout(p);
    const int B = p.B, T = p.T, H = p.H, D = p.D, C = p.C;
    const int64_t BT = (int64_t)B * T;
    const bool do_drop = training && drop > 0.f;
    CUDA_TRY(cudaMemsetAsync(grads, 0, sizeof(float) * p.nparams, st));
    // head: dcat = dlogits lin_w ; dlin_w = dlogits^T cat ; dlin_b = colsum(dlogits)
    GemmArgs a = gemm_args(dlogits, params + p.off_linw(), scratch + W.dcat, B, 3 * H, C, C, 1, 1, 3 * H, 3 * H);
    TRY(sgemm_launch(a, st));
    GemmArgs w = gemm_args(dlogits, stash + S.cat, grads + p.off_linw(), C, 3 * H, B, 1, C, 1, 3 * H, 3 * H);
    TRY(sgemm_launch(w, st));
    TRY(colsum_launch(dlogits, grads + p.off_linb(), B, C, C, 1, 0, 0, st));
    float* dY = scratch + W.dYa;
    float* dYnext = scratch + W.dYb;
    float* dhc = scratch + W.dhc;
    KLAUNCH(KC_HEAD, 0.0, 0.0, st, head_bwd_dy_kernel<<<nblk(BT * H, 256), 256, 0, st>>>(scratch + W.dcat, (const int*)(stash + S.arg), dY, dhc, B, T, H, D));
    for (int l = p.L - 1; l >= 0; --l) {
        const int I = (int)p.in_size(l);
        const float* Y = stash + S.Y[l];
        const float* G = stash + S.G[l];
        const float* h0l = h0 ? h0 + (int64_t)l * D * B * H : nullptr;
        float* dgi = scratch + W.dgi;
        float* dgh = scratch + W.dgh;
        if (l != p.L - 1) CUDA_TRY(cudaMemsetAsync(dhc, 0, sizeof(float) * D * B * H, st));
        for (int s = 0; s < T; ++s) {
            KLAUNCH(KC_GATES_BWD, 0.0, 0.0, st, gru_gates_bwd_kernel<<<nblk((int64_t)D * B * H, 256), 256, 0, st>>>(G, Y, h0l, dY, dhc, dgi, dgh, B, T, H, D, s));
            // dhc[d] += dgh_t[d] W_hh[d]   (rows t: dir0 -> T-1-s, dir1 -> s)
            const int t0 = T - 1 - s, t1 = s;
            GemmArgs r = gemm_args(dgh + (int64_t)t0 * 3 * H, params + p.off_whh(l, 0), dhc, B, H, 3 * H,
                                   (int64_t)T * 3 * H, 1, 1, H, H);
            r.beta = 1; r.batch = D;
            r.zA = BT * 3 * H + (int64_t)(t1 - t0) * 3 * H; r.zB = p.ld_block(l); r.zC = (int64_t)B * H;
            TRY(sgemm_launch(r, st));
        }
        if (dh0) CUDA_TRY(cudaMemcpyAsync(dh0 + (int64_t)l * D * B * H, dhc, sizeof(float) * D * B * H,
                                          cudaMemcpyDeviceToDevice, st));
        // layer input as seen by the projection (dropped copy when dropout was applied)
        const float* inp = l == 0 ? (x ? x : stash + S.X[0]) : stash + S.Y[l - 1];     // x == NULL: forward_windows left it in the stash
        if (do_drop && (l == 0 || p.L > 1)) inp = stash + S.X[l];
        const int splitk = (int)min((int64_t)64, max((int64_t)1, BT / 512));
        for (int d = 0; d < D; ++d) {
            const float* dgi_d = dgi + (int64_t)d * BT * 3 * H;
            const float* dgh_d = dgh + (int64_t)d * BT * 3 * H;
            // dW_ih = dgi^T X
            GemmArgs wi = gemm_args(dgi_d, inp, grads + p.off_wih(l, d), 3 * H, I, (int)BT, 1, 3 * H, 1, I, I);
            wi.splitk = splitk;
            TRY(sgemm_launch(wi, st));
            // dW_hh = dgh^T H_prev ; H_prev(b,t) = Y[b,t-1] (dir 0) / Y[b,t+1] (dir 1), h0 at the first step
            if (T > 1) {
                const float* hp = Y + (int64_t)d * H + (d == 0 ? -(int64_t)D * H : (int64_t)D * H);
                GemmArgs wh = gemm_args(dgh_d, hp, grads + p.off_whh(l, d), 3 * H, H, (int)BT, 1, 3 * H, 1,
                                        (int64_t)D * H, H);
                wh.splitk = splitk; wh.mask_period = T; wh.mask_skip = d == 0 ? 0 : T - 1;
                TRY(sgemm_launch(wh, st));
            }
            if (h0l) {
                const int tf = d == 0 ? 0 : T - 1;
                GemmArgs w0 = gemm_args(dgh_d + (int64_t)tf * 3 * H, h0l + (int64_t)d * B * H, grads + p.off_whh(l, d),
                                        3 * H, H, B, 1, (int64_t)T * 3 * H, 1, H, H);
                w0.splitk = 2;       // forces the atomic-accumulate epilogue onto the existing sums
                TRY(sgemm_launch(w0, st));
            }
            TRY(colsum_launch(dgi_d, grads + p.off_bih(l, d), BT, 3 * H, 3 * H, 1, 0, 0, st));
            TRY(colsum_launch(dgh_d, grads + p.off_bhh(l, d), BT, 3 * H, 3 * H, 1, 0, 0, st));
        }
        // dX = sum_d dgi[d] W_ih[d]
        float* dxo = l == 0 ? dx : dYnext;
        if (dxo) {
            for (int d = 0; d < D; ++d) {
                GemmArgs gx = gemm_args(dgi + (int64_t)d * BT * 3 * H, params + p.off_wih(l, d), dxo, (int)BT, I, 3 * H,
                                        3 * H, 1, 1, I, I);
                gx.beta = d;
                TRY(sgemm_launch(gx, st));
            }
            if (do_drop && (l == 0 || p.L > 1)) {
                // d(dropout): same mask, in place.  dropout_kernel(in=dxo) multiplies by mask/(1-p)
                KLAUNCH(KC_MISC, 0.0, 0.0, st, dropout_kernel<<<148 * 8, 256, 0, st>>>(dxo, dxo, BT * I, T, I, l == 0 ? spatial : 0, drop, seed, (uint32_t)l));
            }
        }
        float* tmp = dY; dY = dYnext; dYnext = tmp;
    }
    return BIGRU_OK;
}

// ------------------------------------------------------------------------------------------
// exported compute entry points
// ------------------------------------------------------------------------------------------
extern "C" int bigru_forward(const bigru_plan* plan, const float* d_params, const float* d_x, const float* d_h0,
                             float dropout_p, int spatial, int training, uint64_t seed, void* d_stash,
                             void* d_scratch, float* d_logits, float* d_hn, void* stream) {
    if (!plan || !d_params || !d_x || !d_stash || !d_scratch || !d_logits) {
        bigru_set_error("forward: null argument");
        return BIGRU_ERR_ARG;
    }
    if (dropout_p < 0.f || dropout_p >= 1.f) { bigru_set_error("forward: dropout_p must be in [0,1)"); return BIGRU_ERR_ARG; }
    cudaStream_t st = (cudaStream_t)stream;
    if (plan->prec == BIGRU_PREC_BF16)
        return forward_bf16(*plan, d_params, d_x, d_h0, dropout_p, spatial, training, seed, d_stash, d_scratch,
                            d_logits, d_hn, st);
    if (plan->prec == BIGRU_PREC_BF16X3)
        return forward_x3(*plan, d_params, d_x, d_h0, dropout_p, spatial, training, seed, d_stash, d_scratch,
                          d_logits, d_hn, st);
    return forward_f32(*plan, d_params, d_x, d_h0, dropout_p, spatial, training, seed, (float*)d_stash,
                       (float*)d_scratch, d_logits, d_hn, st);
}

extern "C" int bigru_backward(const bigru_plan* plan, const float* d_params, const float* d_x, const float* d_h0,
                              float dropout_p, int spatial, int training, uint64_t seed, const void* d_stash,
                              void* d_scratch, const float* d_dlogits, float* d_grads, float* d_dx, float* d_dh0,
                              void* stream) {
    if (!plan || !d_params || !d_stash || !d_scratch || !d_dlogits || !d_grads) {
        bigru_set_error("backward: null argument");
        return BIGRU_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    if (plan->prec == BIGRU_PREC_BF16)
        return backward_bf16(*plan, d_params, d_x, d_h0, dropout_p, spatial, training, seed, d_stash, d_scratch,
                             d_dlogits, d_grads, d_dx, d_dh0, st);
    if (plan->prec == BIGRU_PREC_BF16X3)
        return backward_x3(*plan, d_params, d_x, d_h0, dropout_p, spatial, training, seed, d_stash, d_scratch,
                           d_dlogits, d_grads, d_dx, d_dh0, st);
    return backward_f32(*plan, d_params, d_x, d_h0, dropout_p, spatial, training, seed, (const float*)d_stash,
                        (float*)d_scratch, d_dlogits, d_grads, d_dx, d_dh0, st);
}

extern "C" int bigru_backward_layers(const bigru_plan* plan, const float* d_params, const float* d_x, const float* d_h0,
                                     float dropout_p, int spatial, int training, uint64_t seed, const void* d_stash,
                                     void* d_scratch, const float* d_dlogits, float* d_grads, float* d_dx, float* d_dh0,
                                     int layer_from, int layer_to, void* stream) {
    if (!plan || !d_params || !d_stash || !d_scratch || !d_dlogits || !d_grads) {
        bigru_set_error("backward_layers: null argument");
        return BIGRU_ERR_ARG;
    }
    if (layer_from >= plan->L || layer_to < 0 || layer_to > layer_from) {
        bigru_set_error("backward_layers: bad layer range %d..%d for %d layers", layer_from, layer_to, plan->L);
        return BIGRU_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    if (plan->prec == BIGRU_PREC_BF16)
        return backward_bf16(*plan, d_params, d_x, d_h0, dropout_p, spatial, training, seed, d_stash, d_scratch,
                             d_dlogits, d_grads, d_dx, d_dh0, st, layer_from, layer_to);
    if (plan->prec == BIGRU_PREC_BF16X3)
        return backward_x3(*plan, d_params, d_x, d_h0, dropout_p, spatial, training, seed, d_stash, d_scratch,
                           d_dlogits, d_grads, d_dx, d_dh0, st, layer_from, layer_to);
    bigru_set_error("backward_layers: the fp32 path runs its layers in one call (bigru_backward)");
    return BIGRU_ERR_UNSUPPORTED;
}

extern "C" int bigru_forward_windows(const bigru_plan* plan, const float* d_params, const float* d_src, const float* d_xmin,
                                     const float* d_xmax, int64_t start, int64_t N, float dropout_p, int spatial,
                                     int training, uint64_t seed, void* d_stash, void* d_scratch, float* d_logits,
                                     float* d_hn, void* stream) {
    if (!plan || !d_params || !d_src || !d_stash || !d_scratch || !d_logits || ((d_xmin == nullptr) != (d_xmax == nullptr))) {
        bigru_set_error("forward_windows: null argument");
        return BIGRU_ERR_ARG;
    }
    if (start < 0 || start + plan->B + plan->T - 1 > N) {
        bigru_set_error("forward_windows: windows [%lld, %lld) exceed the %lld-row chunk", (long long)start,
                        (long long)(start + plan->B + plan->T - 1), (long long)N);
        return BIGRU_ERR_ARG;
    }
    if (dropout_p < 0.f || dropout_p >= 1.f) { bigru_set_error("forward_windows: dropout_p must be in [0,1)"); return BIGRU_ERR_ARG; }
    cudaStream_t st = (cudaStream_t)stream;
    if (plan->prec == BIGRU_PREC_BF16)
        return forward_bf16(*plan, d_params, nullptr, nullptr, dropout_p, spatial, training, seed, d_stash, d_scratch,
                            d_logits, d_hn, st, WindowSrc{d_src, d_xmin, d_xmax, start});
    if (plan->prec == BIGRU_PREC_BF16X3)
        return forward_x3(*plan, d_params, nullptr, nullptr, dropout_p, spatial, training, seed, d_stash, d_scratch,
                          d_logits, d_hn, st, WindowSrc{d_src, d_xmin, d_xmax, start});
    // fp32 path: collate into the stash slot of the layer-0 input, then the ordinary forward
    float* xw = (float*)d_stash + stash_layout(*plan).X[0];
    TRY(bigru_window_gather_norm(d_src, d_xmin, d_xmax, start, N, plan->B, plan->T, plan->F, xw, stream));
    return forward_f32(*plan, d_params, xw, nullptr, dropout_p, spatial, training, seed, (float*)d_stash,
                       (float*)d_scratch, d_logits, d_hn, st);
}

extern "C" int bigru_chunk_minmax(const float* d_table, int64_t N, int F, int64_t row_lo, int64_t row_hi, float* d_min,
                                  float* d_max, void* stream) {
    if (!d_table || !d_min || !d_max || F <= 0 || row_lo < 0 || row_hi > N || row_lo >= row_hi) {
        bigru_set_error("chunk_minmax: bad argument");
        return BIGRU_ERR_ARG;
    }
    KLAUNCH(KC_GATHER, 0.0, 4.0 * (row_hi - row_lo) * F, (cudaStream_t)stream,
            chunk_minmax_kernel<<<(F + 31) / 32, dim3(32, 8), 0, (cudaStream_t)stream>>>(d_table, F, row_lo, row_hi, d_min, d_max));
    return BIGRU_OK;
}

extern "C" int bigru_window_features(const float* d_close, const float* d_high, const float* d_low, const float* d_volume,
                                     const float* d_delta, int64_t n, const int* vol_periods, int n_vol, const int* price_periods,
                                     int n_price, const int* delta_periods, int n_delta, int bb_period, float bb_std, int stochastic,
                                     float n1, float n2, float* d_out, float* d_targets, int* n_out, void* stream) {
    if (n_vol < 0 || n_vol > 8 || n_price < 0 || n_price > 8 || n_delta < 0 || n_delta > 8 || bb_period < 0 || n < 0 ||
        (n_vol && !vol_periods) || (n_price && !price_periods) || (n_delta && !delta_periods)) {
        bigru_set_error("window_features: bad argument (at most 8 periods per list)");
        return BIGRU_ERR_ARG;
    }
    FeatureCfg cfg{};
    cfg.n_vol = n_vol; cfg.n_price = n_price; cfg.n_delta = n_delta;
    for (int i = 0; i < n_vol; ++i) cfg.vol_p[i] = vol_periods[i];
    for (int i = 0; i < n_price; ++i) cfg.price_p[i] = price_periods[i];
    for (int i = 0; i < n_delta; ++i) cfg.delta_p[i] = delta_periods[i];
    for (int i = 0; i < 8; ++i)
        if ((i < n_vol && cfg.vol_p[i] < 1) || (i < n_price && cfg.price_p[i] < 1) || (i < n_delta && cfg.delta_p[i] < 1)) {
            bigru_set_error("window_features: periods must be >= 1");
            return BIGRU_ERR_ARG;
        }
    cfg.bb_period = bb_period; cfg.bb_std = bb_std; cfg.stochastic = stochastic ? 1 : 0; cfg.n1 = n1; cfg.n2 = n2;
    cfg.n_out = (bb_period > 0 ? 2 : 0) + n_vol + n_price + n_delta + (stochastic ? 1 : 0) + 2;
    if (n_out) *n_out = cfg.n_out;
    if (!d_out || n == 0) return BIGRU_OK;
    if (!d_close || !d_high || !d_low || (n_vol && !d_volume) || (n_delta && !d_delta)) {
        bigru_set_error("window_features: null column");
        return BIGRU_ERR_ARG;
    }
    int halo = 14;
    for (int i = 0; i < n_vol; ++i) halo = std::max(halo, cfg.vol_p[i] - 1);
    for (int i = 0; i < n_price; ++i) halo = std::max(halo, cfg.price_p[i] - 1);
    for (int i = 0; i < n_delta; ++i) halo = std::max(halo, cfg.delta_p[i] - 1);
    halo = std::max(halo, bb_period - 1);
    if (halo > 4095) { bigru_set_error("window_features: periods above 4096 rows are not supported"); return BIGRU_ERR_UNSUPPORTED; }
    const int span = FEAT_TR + halo;
    const size_t smem = sizeof(float) * ((size_t)4 * span + 16 + (size_t)FEAT_TR * (cfg.n_out + 4));
    // the reference's own configuration (config.py:40-49) runs with compile-time periods
    const bool fast = n_vol == 2 && cfg.vol_p[0] == 6 && cfg.vol_p[1] == 20 && n_price == 1 && cfg.price_p[0] == 20 && n_delta == 1 &&
                      cfg.delta_p[0] == 12 && bb_period == 20 && stochastic;
    if (smem > 48 * 1024)        // per-device opt-in, set on every call (no process-wide cache: a second GPU would miss it)
        CUDA_TRY(fast ? cudaFuncSetAttribute(window_features_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                      : cudaFuncSetAttribute(window_features_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const unsigned blocks = (unsigned)std::min<int64_t>((n + FEAT_TR - 1) / FEAT_TR, 148 * 8);
    if (fast)
        KLAUNCH(KC_GATHER, 0.0, 4.0 * n * (5 + cfg.n_out + 4), (cudaStream_t)stream,
                window_features_kernel<true><<<blocks, FEAT_TR, smem, (cudaStream_t)stream>>>(d_close, d_high, d_low, d_volume, d_delta, n, cfg,
                                                                                              halo, d_out, d_targets));
    else
        KLAUNCH(KC_GATHER, 0.0, 4.0 * n * (5 + cfg.n_out + 4), (cudaStream_t)stream,
                window_features_kernel<false><<<blocks, FEAT_TR, smem, (cudaStream_t)stream>>>(d_close, d_high, d_low, d_volume, d_delta, n, cfg,
                                                                                               halo, d_out, d_targets));
    return BIGRU_OK;
}

extern "C" int bigru_infer_window(const float* d_params, const float* d_x, const float* d_xmin, const float* d_xmax, int B, int T,
                                  int F, int H, int L, int C, int bidirectional, float* d_logits, float* d_probs, void* stream) {
    if (!d_params || !d_x || !d_logits || B <= 0 || T <= 0 || F <= 0 || H <= 0 || L <= 0 || C <= 0 || ((d_xmin == nullptr) != (d_xmax == nullptr))) {
        bigru_set_error("infer_window: bad argument");
        return BIGRU_ERR_ARG;
    }
    const int D = bidirectional ? 2 : 1, DH = D * H, W = F > DH ? F : DH;
    const size_t smem = sizeof(float) * ((size_t)T * W + (size_t)T * DH + 2 * (size_t)DH + 3 * (size_t)H);
    if (DH > 1024 || smem > 200 * 1024) {
        bigru_set_error("infer_window: window too large for the single-CTA path (D*H=%d, %zu bytes of shared memory); use bigru_forward", DH, smem);
        return BIGRU_ERR_UNSUPPORTED;
    }
    if (smem > 48 * 1024)
        CUDA_TRY(cudaFuncSetAttribute(infer_window_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int threads = std::max(32, ((DH + 31) / 32) * 32);
    KLAUNCH(KC_MISC, 0.0, 0.0, (cudaStream_t)stream,
            infer_window_kernel<<<B, threads, smem, (cudaStream_t)stream>>>(d_params, d_x, d_xmin, d_xmax, T, F, H, L, C, D, d_logits, d_probs));
    return BIGRU_OK;
}

// ------------------------------------------------------------------------------------------
// cluster-resident live inference (csrc/infer_cluster.cuh).  Workspace in floats, each region 256-byte aligned:
// normalised input [B*T*F] | gi [D][B*T][3H] | layer output Y [B][T][D*H] (reused by every layer: a layer's projection
// has consumed its input before its scan overwrites it).
// ------------------------------------------------------------------------------------------
struct InferWork { int64_t xn, gi, y, total; };
static InferWork infer_work_layout(int B, int T, int F, int H, int D) {
    auto al = [](int64_t n) { return (n + 63) / 64 * 64; };
    const int64_t BT = (int64_t)B * T;
    InferWork w{};
    w.xn = 0;
    w.gi = w.xn + al(BT * F);
    w.y = w.gi + al((int64_t)D * BT * 3 * H);
    w.total = w.y + al(BT * D * H);
    return w;
}

static bool infer_cluster_shape_ok(int B, int T, int F, int H, int L, int C) {
    return B > 0 && T > 0 && F > 0 && H > 0 && L > 0 && C > 0;
}

extern "C" int bigru_infer_cluster_workspace_bytes(int B, int T, int F, int H, int L, int bidirectional, size_t* bytes) {
    if (!bytes || !infer_cluster_shape_ok(B, T, F, H, L, 1)) {
        bigru_set_error("infer_cluster_workspace_bytes: bad argument");
        return BIGRU_ERR_ARG;
    }
    *bytes = (size_t)infer_work_layout(B, T, F, H, bidirectional ? 2 : 1).total * sizeof(float);
    return BIGRU_OK;
}

// Cluster geometry: U units per CTA (a multiple of 4, at most 32), NC = ceil(H / U) CTAs.  The per-step time is bound by the
// shared-memory reads of the W_hh slice (3*U*Hp*4 bytes per CTA), so the widest cluster wins: up to 16 CTAs
// (non-portable) where the device grants them, else 8.  BIGRU_INFER_CLUSTER_CTAS (8 or 16) caps it for measurement.
// G windows per cluster: the smallest power of two <= 4 that covers B (capped by shared memory; G = 8 spills registers).
struct InferGeo { int NC, U, Hp, G; size_t smem; };
static InferGeo infer_geometry(int B, int H, int max_nc) {
    InferGeo g{};
    g.U = (int)((cdiv64(H, max_nc) + 3) / 4 * 4);
    g.NC = (int)cdiv64(H, g.U);
    g.Hp = g.NC * g.U;
    g.G = 1;
    while (g.G < 4 && g.G < B) g.G *= 2;
    while (g.G > 1 && icl::scan_smem_bytes(g.U, g.Hp, g.G) > 227 * 1024) g.G /= 2;
    g.smem = icl::scan_smem_bytes(g.U, g.Hp, g.G);
    return g;
}

template <int G>
static int infer_scan_launch(const InferGeo& geo, int ngroups, int D, const float* gi, const float* w_hh, const float* b_hh,
                             int64_t dir_stride, float* Y, int B, int T, int H, cudaStream_t st, bool probe, int* max_clusters) {
    auto kern = icl::infer_cluster_scan_kernel<G>;
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)geo.smem));
    if (geo.NC > 8) CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(geo.NC, ngroups, D);
    cfg.blockDim = dim3(icl::kThreads);
    cfg.dynamicSmemBytes = geo.smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = geo.NC; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    if (probe) {
        int n = 0;
        cudaError_t e = cudaOccupancyMaxActiveClusters(&n, kern, &cfg);
        if (e != cudaSuccess) { cudaGetLastError(); n = 0; }
        *max_clusters = n;
        return BIGRU_OK;
    }
    KLAUNCH(KC_INFER, 0.0, 0.0, st, CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, gi, w_hh, b_hh, dir_stride, Y, B, T, H, D, geo.U)));
    return BIGRU_OK;
}

static int infer_scan_dispatch(const InferGeo& geo, int ngroups, int D, const float* gi, const float* w_hh, const float* b_hh,
                               int64_t dir_stride, float* Y, int B, int T, int H, cudaStream_t st, bool probe, int* max_clusters) {
    switch (geo.G) {
        case 1: return infer_scan_launch<1>(geo, ngroups, D, gi, w_hh, b_hh, dir_stride, Y, B, T, H, st, probe, max_clusters);
        case 2: return infer_scan_launch<2>(geo, ngroups, D, gi, w_hh, b_hh, dir_stride, Y, B, T, H, st, probe, max_clusters);
        default: return infer_scan_launch<4>(geo, ngroups, D, gi, w_hh, b_hh, dir_stride, Y, B, T, H, st, probe, max_clusters);
    }
}

// the widest cluster the device grants at this shared-memory size (opt-ins set on every call); *granted is
// cudaOccupancyMaxActiveClusters of the chosen launch
static int infer_pick_geometry(int B, int H, int D, InferGeo* out, int* granted) {
    if (H > icl::kMaxHidden) {
        bigru_set_error("infer_cluster: hidden size %d above %d (16 CTAs x 32 units) is not supported", H, icl::kMaxHidden);
        return BIGRU_ERR_UNSUPPORTED;
    }
    int cap = icl::kMaxCluster;
    if (const char* e = getenv("BIGRU_INFER_CLUSTER_CTAS")) cap = atoi(e) == 8 ? 8 : icl::kMaxCluster;
    InferGeo geo = infer_geometry(B, H, cap);
    *granted = 0;
    TRY(infer_scan_dispatch(geo, (int)cdiv64(B, geo.G), D, nullptr, nullptr, nullptr, 0, nullptr, B, 1, H, nullptr, true, granted));
    if (*granted <= 0 && geo.NC > 8) {
        const int nc16 = geo.NC;
        geo = infer_geometry(B, H, 8);
        if (geo.U > icl::kMaxUnits) {
            bigru_set_error("infer_cluster: hidden size %d needs a %d-CTA cluster, which this device does not grant; "
                            "8-CTA clusters hold H <= %d", H, nc16, 8 * icl::kMaxUnits);
            return BIGRU_ERR_UNSUPPORTED;
        }
        TRY(infer_scan_dispatch(geo, (int)cdiv64(B, geo.G), D, nullptr, nullptr, nullptr, 0, nullptr, B, 1, H, nullptr, true, granted));
    }
    if (*granted <= 0) {
        bigru_set_error("infer_cluster: the device grants no %d-CTA cluster with %zu bytes of shared memory per CTA", geo.NC, geo.smem);
        return BIGRU_ERR_UNSUPPORTED;
    }
    *out = geo;
    return BIGRU_OK;
}

extern "C" int bigru_infer_cluster_geometry(int B, int H, int bidirectional, int* cluster_ctas, int* units_per_cta,
                                            int* windows_per_cluster, int* max_active_clusters) {
    if (B <= 0 || H <= 0 || !cluster_ctas || !units_per_cta || !windows_per_cluster || !max_active_clusters) {
        bigru_set_error("infer_cluster_geometry: bad argument");
        return BIGRU_ERR_ARG;
    }
    InferGeo geo;
    TRY(infer_pick_geometry(B, H, bidirectional ? 2 : 1, &geo, max_active_clusters));
    *cluster_ctas = geo.NC; *units_per_cta = geo.U; *windows_per_cluster = geo.G;
    return BIGRU_OK;
}

extern "C" int bigru_infer_cluster(const float* d_params, const float* d_x, const float* d_xmin, const float* d_xmax, int B, int T,
                                   int F, int H, int L, int C, int bidirectional, void* d_work, float* d_logits, float* d_probs,
                                   void* stream) {
    if (!d_params || !d_x || !d_work || !d_logits || !infer_cluster_shape_ok(B, T, F, H, L, C) || L > 16 ||
        ((d_xmin == nullptr) != (d_xmax == nullptr)) || ((uintptr_t)d_work & 15)) {
        bigru_set_error("infer_cluster: bad argument");
        return BIGRU_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int D = bidirectional ? 2 : 1;
    InferGeo geo;
    int granted = 0;
    TRY(infer_pick_geometry(B, H, D, &geo, &granted));
    const int ngroups = (int)cdiv64(B, geo.G);
    bigru_plan p{};
    p.B = B; p.T = T; p.F = F; p.H = H; p.L = L; p.C = C; p.D = D;
    const InferWork w = infer_work_layout(B, T, F, H, D);
    float* work = (float*)d_work;
    const int64_t BT = (int64_t)B * T;
    const float* inp = d_x;
    if (d_xmin) {
        // (x - min) / (max - min) of every row: the window gather over B*T consecutive rows
        float* xn = work + w.xn;
        const unsigned blocks = (unsigned)std::min<int64_t>(cdiv64(BT * F, 256), 148 * 8);
        KLAUNCH(KC_GATHER, 0.0, 8.0 * BT * F, st, window_gather_kernel<1><<<blocks, 256, 0, st>>>(d_x, d_xmin, d_xmax, 0, 1, (int)BT, F, xn));
        inp = xn;
    }
    float* Y = work + w.y;
    for (int l = 0; l < L; ++l) {
        const int I = (int)p.in_size(l);
        GemmArgs g = gemm_args(inp, d_params + p.off_wih(l, 0), work + w.gi, (int)BT, 3 * H, I, I, 1, I, 1, 3 * H);
        g.bias = d_params + p.off_bih(l, 0);
        g.batch = D; g.zA = 0; g.zB = p.ld_block(l); g.zBias = p.ld_block(l); g.zC = BT * 3 * H;
        TRY(sgemm_launch(g, st));
        TRY(infer_scan_dispatch(geo, ngroups, D, work + w.gi, d_params + p.off_whh(l, 0), d_params + p.off_bhh(l, 0), p.ld_block(l), Y,
                                B, T, H, st, false, nullptr));
        inp = Y;
    }
    KLAUNCH(KC_HEAD, 0.0, 0.0, st,
            icl::infer_head_kernel<<<B, 128, 3 * H * sizeof(float), st>>>(Y, d_params + p.off_linw(), T, H, C, D, d_logits, d_probs));
    return BIGRU_OK;
}

extern "C" int bigru_loss(int kind, const float* d_logits, const void* d_target, const float* d_weight,
                          const float* d_pos_weight, int B, int C, double denom, float* d_loss, float* d_dlogits,
                          void* stream) {
    if (!d_logits || !d_target || !d_loss || B <= 0 || C <= 0 || denom <= 0 || kind < 0 || kind > 2) {
        bigru_set_error("loss: bad argument");
        return BIGRU_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaMemsetAsync(d_loss, 0, sizeof(float), st));
    if (kind == BIGRU_LOSS_MLSM) { d_weight = nullptr; d_pos_weight = nullptr; }
    KLAUNCH(KC_LOSS, 0.0, 0.0, st, loss_kernel<<<nblk(B, 128), 128, 0, st>>>(kind, d_logits, d_target, d_weight, d_pos_weight, B, C,
                                             (float)(1.0 / denom), d_loss, d_dlogits));
    return BIGRU_OK;
}

extern "C" int bigru_sqnorm(const float* d_g, int64_t n, float* d_out, void* stream) {
    if (!d_g || !d_out || n < 0) { bigru_set_error("sqnorm: bad argument"); return BIGRU_ERR_ARG; }
    if (n == 0) return BIGRU_OK;
    const unsigned blocks = (unsigned)min((int64_t)148 * 4, cdiv64(n, 256));
    KLAUNCH(KC_OPTIM, 0.0, 0.0, (cudaStream_t)stream, sqnorm_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(d_g, n, d_out));
    return BIGRU_OK;
}

extern "C" int bigru_clip_adam_step(float* d_params, float* d_grads, float* d_m, float* d_v, int64_t n,
                                    const float* d_sqnorm, float clip, float lr, float b1, float b2, float eps,
                                    int step, float grad_scale, void* stream) {
    if (!d_params || !d_grads || !d_m || !d_v || !d_sqnorm || n <= 0 || step < 1) {
        bigru_set_error("clip_adam_step: bad argument");
        return BIGRU_ERR_ARG;
    }
    const double bc1 = 1.0 - pow((double)b1, step), bc2 = 1.0 - pow((double)b2, step);
    const unsigned blocks = (unsigned)min((int64_t)148 * 8, cdiv64(n, 256));
    KLAUNCH(KC_OPTIM, 0.0, 0.0, (cudaStream_t)stream, clip_adam_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(d_params, d_grads, d_m, d_v, n, d_sqnorm, clip, lr, b1,
                                                                b2, eps, (float)bc1, (float)sqrt(bc2), grad_scale));
    return BIGRU_OK;
}

extern "C" int bigru_adam_tick(int* d_step, float* d_sqnorm, void* stream) {
    if (!d_step || !d_sqnorm) { bigru_set_error("adam_tick: null argument"); return BIGRU_ERR_ARG; }
    KLAUNCH(KC_OPTIM, 0.0, 0.0, (cudaStream_t)stream, adam_tick_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(d_step, d_sqnorm));
    return BIGRU_OK;
}

extern "C" int bigru_clip_adam_step_dev(float* d_params, float* d_grads, float* d_m, float* d_v, int64_t n,
                                        const float* d_sqnorm, float clip, float lr, float b1, float b2, float eps,
                                        const int* d_step, float grad_scale, void* stream) {
    if (!d_params || !d_grads || !d_m || !d_v || !d_sqnorm || !d_step || n <= 0) {
        bigru_set_error("clip_adam_step_dev: bad argument");
        return BIGRU_ERR_ARG;
    }
    const unsigned blocks = (unsigned)min((int64_t)148 * 8, cdiv64(n, 256));
    KLAUNCH(KC_OPTIM, 0.0, 0.0, (cudaStream_t)stream, clip_adam_dev_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(d_params, d_grads, d_m, d_v, n, d_sqnorm, clip,
                                                                    lr, b1, b2, eps, d_step, grad_scale));
    return BIGRU_OK;
}

extern "C" int bigru_window_gather_norm(const float* d_src, const float* d_xmin, const float* d_xmax, int64_t start,
                                        int64_t N, int B, int T, int F, float* d_out, void* stream) {
    if (B == 0 && T > 0 && F > 0 && start >= 0) return BIGRU_OK;          // empty batch: nothing to write
    if (!d_src || !d_out || B < 0 || T <= 0 || F <= 0 || start < 0 || (B > 0 && start + B + T - 1 > N) ||
        ((d_xmin == nullptr) != (d_xmax == nullptr))) {
        bigru_set_error("window_gather_norm: bad argument (start=%lld B=%d T=%d N=%lld)", (long long)start, B, T, (long long)N);
        return BIGRU_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const bool vec = F % 4 == 0 && ((uintptr_t)d_src % 16 == 0) && ((uintptr_t)d_out % 16 == 0) &&
                     (!d_xmin || (((uintptr_t)d_xmin % 16 == 0) && ((uintptr_t)d_xmax % 16 == 0)));
    const int64_t total = (int64_t)B * T * (vec ? F / 4 : F);
    const unsigned blocks = (unsigned)min((int64_t)148 * 16, cdiv64(total, 256));
    // algorithmic bytes: write B*T*F floats, read the (B+T-1)*F source rows once (SURVEY.md 8(d))
    const double bytes = 4.0 * ((double)B * T * F + (double)(B + T - 1) * F);
    if (vec) KLAUNCH(KC_GATHER, 0.0, bytes, st, window_gather_kernel<4><<<blocks, 256, 0, st>>>(d_src, d_xmin, d_xmax, start, B, T, F, d_out));
    else KLAUNCH(KC_GATHER, 0.0, bytes, st, window_gather_kernel<1><<<blocks, 256, 0, st>>>(d_src, d_xmin, d_xmax, start, B, T, F, d_out));
    return BIGRU_OK;
}

extern "C" int bigru_window_targets(const float* d_y, int64_t start, int64_t N, int B, int T, int C, float* d_out,
                                    void* stream) {
    if (B == 0 && T > 0 && C > 0 && start >= 0) return BIGRU_OK;
    if (!d_y || !d_out || B < 0 || T <= 0 || C <= 0 || start < 0 || (B > 0 && start + B + T - 1 > N)) {
        bigru_set_error("window_targets: bad argument");
        return BIGRU_ERR_ARG;
    }
    if (B == 0) return BIGRU_OK;
    KLAUNCH(KC_GATHER, 0.0, 0.0, (cudaStream_t)stream, window_targets_kernel<<<nblk((int64_t)B * C, 256), 256, 0, (cudaStream_t)stream>>>(d_y, start, B, T, C, d_out));
    return BIGRU_OK;
}

extern "C" int bigru_multilabel_counts(const float* d_logits, const float* d_target, int B, int C,
                                       long long* d_counts, void* stream) {
    if (!d_logits || !d_target || !d_counts || B <= 0 || C <= 0) { bigru_set_error("multilabel_counts: bad argument"); return BIGRU_ERR_ARG; }
    KLAUNCH(KC_MISC, 0.0, 0.0, (cudaStream_t)stream, multilabel_counts_kernel<<<nblk(B, 128), 128, 0, (cudaStream_t)stream>>>(d_logits, d_target, B, C,
                                                                            (unsigned long long*)d_counts));
    return BIGRU_OK;
}

// ------------------------------------------------------------------------------------------
// measurement hooks (bench.py): launch counter and per-kernel-class CUDA-event timing
// ------------------------------------------------------------------------------------------
extern "C" long long bigru_launch_count(void) { return profiler().launches.load(); }
// kernels replayed through a captured CUDA graph do not pass the launch macros: the caller reports them (n per replay)
extern "C" void bigru_launch_count_add(long long n) { profiler().launches.fetch_add(n, std::memory_order_relaxed); }

extern "C" int bigru_prof_enable(int on) {
    Profiler& p = profiler();
    std::lock_guard<std::mutex> g(p.mu);
    for (auto& r : p.recs) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    p.recs.clear();
    p.enabled.store(on ? 1 : 0);
    return BIGRU_OK;
}

extern "C" int bigru_prof_classes(void) { return KC_COUNT; }
extern "C" const char* bigru_prof_class_name(int cls) { return cls >= 0 && cls < KC_COUNT ? kKClassNames[cls] : ""; }

// Sums the recorded launches of class `cls` (synchronises on their events).
extern "C" int bigru_prof_report(int cls, double* ms, long long* launches, double* flops, double* bytes) {
    if (cls < 0 || cls >= KC_COUNT || !ms || !launches || !flops || !bytes) { bigru_set_error("prof_report: bad argument"); return BIGRU_ERR_ARG; }
    Profiler& p = profiler();
    std::lock_guard<std::mutex> g(p.mu);
    *ms = 0; *launches = 0; *flops = 0; *bytes = 0;
    for (auto& r : p.recs) {
        if (r.cls != cls) continue;
        CUDA_TRY(cudaEventSynchronize(r.b));
        float t = 0.f;
        CUDA_TRY(cudaEventElapsedTime(&t, r.a, r.b));
        *ms += t; *launches += 1; *flops += r.flops; *bytes += r.bytes;
    }
    return BIGRU_OK;
}
