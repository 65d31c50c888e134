// extern "C" entry points of libb200vad.so (declared in include/b200vad.h).
#include "kernels.cuh"
#include "../../include/b200vad.h"
#include <stdarg.h>
#include <string.h>
#include <stdlib.h>
#include <algorithm>
#include <cmath>
#include <atomic>
#include <mutex>
#include <utility>
#include <vector>

namespace b200vad {

static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

static std::atomic<long long> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

static bool g_prof_on = false;
struct ProfRec { cudaEvent_t a, b; int kind; };
static std::vector<ProfRec> g_prof_events;
static size_t g_prof_used = 0;
static std::mutex g_prof_mu;
void prof_begin(int kind, cudaStream_t st) {
    if (!g_prof_on) return;
    std::lock_guard<std::mutex> lk(g_prof_mu);
    if (g_prof_used == g_prof_events.size()) {
        ProfRec r;
        cudaEventCreate(&r.a);
        cudaEventCreate(&r.b);
        r.kind = 0;
        g_prof_events.push_back(r);
    }
    g_prof_events[g_prof_used].kind = kind;
    cudaEventRecord(g_prof_events[g_prof_used].a, st);
}
void prof_end(int kind, cudaStream_t st) {
    if (!g_prof_on) return;
    std::lock_guard<std::mutex> lk(g_prof_mu);
    (void)kind;
    cudaEventRecord(g_prof_events[g_prof_used].b, st);
    ++g_prof_used;
}

int set_max_dynamic_smem(const void* func, int bytes) {
    static std::mutex mu;
    static std::vector<std::pair<const void*, int>> done[64];          // per device: (kernel, bytes already granted)
    int dev = 0;
    B200VAD_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lk(mu);
    if (dev >= 0 && dev < 64)
        for (auto& e : done[dev])
            if (e.first == func && e.second >= bytes) return B200VAD_OK;
    B200VAD_CUDA(cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    if (dev >= 0 && dev < 64) done[dev].push_back({func, bytes});
    return B200VAD_OK;
}

static int g_impl = 2;        // 2 = tcgen05 kernels (default), 1 = warp-MMA kernels (validation only)
static int g_proj_terms = 2;  // fp16 products per k-step of the layer >= 1 input projections: 2 (default) or 3 (validation)
static int g_head_fused = 1;   // head as one kernel (z1 planes stay on chip, default) or as two launches (validation)
// layers with D <= 256: 2 = fused projection + recurrence with cta_group::2 MMAs on CTA pairs (lstm_pair.cu), 1 = the same on
// single-CTA MMAs (lstm_fused.cu), 0 = projection GEMM -> xg -> recurrence; -1 = not chosen yet (B200VAD_LSTM_MODE, else the default)
static int g_lstm_fused = -1;
static int lstm_mode() {
    if (g_lstm_fused < 0) {
        const char* e = getenv("B200VAD_LSTM_MODE");
        g_lstm_fused = (e && atoi(e) >= 0 && atoi(e) <= 2) ? atoi(e) : 1;
    }
    return g_lstm_fused;
}
static int g_proj_kernel = 2;  // input projections with K <= 256: 0 = gemm_ts_kernel<3>, 1 = gemm_xg2_kernel, 2 = gemm_xg_pair_kernel (default)
static int num_sms_cached() {
    static int n = 0;
    if (!n) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (n <= 0) n = 148;
    }
    return n;
}

static inline size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }
static inline int round64(int k) { return (k + 63) / 64 * 64; }

// ---------------------------------------------------------------- packed model layout
struct LayerOff {
    size_t wih_hi, wih_lo, bias, whh, whh_lo;
    int D, Kp;
};
struct ModelLayout {
    std::vector<LayerOff> layers;
    size_t w1_hi, w1_lo, b1, w2_hi, w2_lo, b2, wc, bc, total;
};
static ModelLayout model_layout(int D, int L) {
    ModelLayout m;
    size_t off = 0;
    for (int l = 0; l < L; ++l) {
        LayerOff o;
        o.D = (l == 0) ? D : 2 * kHidden;
        o.Kp = round64(o.D);
        o.wih_hi = off; off = align_up(off + sizeof(__half) * 2 * kGates * o.Kp);
        o.wih_lo = off; off = align_up(off + sizeof(__half) * 2 * kGates * o.Kp);
        o.bias = off;   off = align_up(off + sizeof(float) * 2 * kGates);
        o.whh = off;    off = align_up(off + sizeof(__half) * 2 * kGates * kHidden);
        o.whh_lo = off; off = align_up(off + sizeof(__half) * 2 * kGates * kHidden);
        m.layers.push_back(o);
    }
    m.w1_hi = off; off = align_up(off + sizeof(__half) * kHidden * 2 * kHidden);
    m.w1_lo = off; off = align_up(off + sizeof(__half) * kHidden * 2 * kHidden);
    m.b1 = off;    off = align_up(off + sizeof(float) * kHidden);
    m.w2_hi = off; off = align_up(off + sizeof(__half) * kHidden * kHidden);
    m.w2_lo = off; off = align_up(off + sizeof(__half) * kHidden * kHidden);
    m.b2 = off;    off = align_up(off + sizeof(float) * kHidden);
    m.wc = off;    off = align_up(off + sizeof(float) * kHidden);
    m.bc = off;    off = align_up(off + sizeof(float));
    m.total = off;
    return m;
}

// Workspace per (sequence, frame): xg fp32 [1024] + two layer buffers of 1024 bytes each (either a
// fp32 [256] row or the fp16 hi / lo planes [256] + [256]) + the fp16 hi / lo planes of the layer-0 input.
// xg is laid out in blocks of 64 sequences (lstm_tc.cu), so sequence counts are rounded up to 64.
static inline size_t round8(size_t d) { return (d + 7) / 8 * 8; }
static inline size_t model_bytes_per_frame(int D) {
    return sizeof(float) * 2 * kGates + 2 * sizeof(float) * 2 * kHidden + 2 * sizeof(__half) * round8(D);
}
static inline size_t model_per_row(int D, int64_t T) { return align_up((size_t)T * model_bytes_per_frame(D)) + 1536; }
static inline int64_t ceil64(int64_t b) { return (b + 63) / 64 * 64; }

static int head_forward(const ModelLayout& m, const char* pk, const float* y, int64_t rows, float* z1, float* z2, float* prob,
                        cudaStream_t st) {
    // Linear(256,128)+lrelu -> Linear(128,128)+lrelu -> Linear(128,1)+sigmoid (PyanNet2.py:183-187)
    GemmArgs g;
    g.A = y; g.lda = 2 * kHidden; g.rows_per_batch = rows; g.a_batch_stride = 0; g.M = rows;
    g.N = kHidden; g.K = 2 * kHidden; g.Kp = 2 * kHidden;
    g.W_hi = reinterpret_cast<const __half*>(pk + m.w1_hi); g.W_lo = reinterpret_cast<const __half*>(pk + m.w1_lo);
    g.bias = reinterpret_cast<const float*>(pk + m.b1);
    g.C = z1; g.ldc = kHidden; g.c_half = 0; g.act = 1;
    int rc = gemm_launch(g, 0, 3, st);
    if (rc) return rc;
    g.A = z1; g.lda = kHidden; g.K = kHidden; g.Kp = kHidden;
    g.W_hi = reinterpret_cast<const __half*>(pk + m.w2_hi); g.W_lo = reinterpret_cast<const __half*>(pk + m.w2_lo);
    g.bias = reinterpret_cast<const float*>(pk + m.b2);
    g.C = z2;
    rc = gemm_launch(g, 0, 3, st);
    if (rc) return rc;
    return classifier_launch(z2, rows, reinterpret_cast<const float*>(pk + m.wc), reinterpret_cast<const float*>(pk + m.bc), prob, st);
}

// x: (B, T, D) fp32, or null with the layer-0 input already split into fp16 planes xp_hi / xp_lo (B, T, round8(D)) whose
// padding channels are zero (the fused fbank: D = 80; the SincNet front end: D = 60, pitch 64)
static int model_forward(const void* packed, int D, int L, const float* x, const __half* xp_hi, const __half* xp_lo, int B,
                         int64_t T, float* prob, void* ws, size_t ws_bytes, cudaStream_t st) {
    B200VAD_CHECK_ARG(packed && (x || (xp_hi && xp_lo && g_impl == 2)) && prob && ws, "null pointer");
    B200VAD_CHECK_ARG(D > 0 && L > 0 && B >= 0 && T >= 0, "bad shape");
    B200VAD_CHECK_ARG(D <= B200VAD_MAX_INPUT_DIM, "input width D > 768 (the widest supported input, B200VAD_MAX_INPUT_DIM)");
    B200VAD_CHECK_ARG((reinterpret_cast<uintptr_t>(ws) & 255) == 0, "workspace must be 256-byte aligned");
    if (B == 0 || T == 0) return B200VAD_OK;
    B200VAD_CHECK_ARG(T < (1 << 24), "T too large");
    const ModelLayout m = model_layout(D, L);
    const char* pk = reinterpret_cast<const char*>(packed);
    const size_t per_row = model_per_row(D, T);
    int64_t Bc = (int64_t)(ws_bytes / per_row) / 64 * 64;       // whole 64-sequence blocks (recurrent CTAs, xg records)
    if (g_impl == 1) Bc = std::min<int64_t>(Bc, std::max<int64_t>(64, (int64_t)(65000LL * 128 / T) / 64 * 64));   // warp-MMA GEMM grid limit
    Bc = std::min<int64_t>(Bc, ceil64(B));
    if (Bc < 64) {
        set_error("model_forward: workspace too small (%zu bytes; need >= %zu = 64 sequences)", ws_bytes, 64 * per_row);
        return B200VAD_ENOMEM;
    }
    const int D8 = (int)round8(D);
    const int sms = num_sms_cached();
    for (int64_t b0 = 0; b0 < B; b0 += Bc) {
        const int bc = (int)std::min<int64_t>(Bc, B - b0);
        const int64_t rows = (int64_t)bc * T;
        char* w = reinterpret_cast<char*>(ws);
        float* xg = reinterpret_cast<float*>(w);                 w += align_up(sizeof(float) * 2 * kGates * ceil64(bc) * T);
        char* buf0 = w;                                          w += align_up(sizeof(float) * 2 * kHidden * rows);
        char* buf1 = w;                                          w += align_up(sizeof(float) * 2 * kHidden * rows);
        __half* x_hi = reinterpret_cast<__half*>(w);             w += align_up(sizeof(__half) * D8 * rows);
        __half* x_lo = reinterpret_cast<__half*>(w);
        const float* xin = x ? x + b0 * T * D : nullptr;
        int rc;
        if (g_impl == 1) {
            // ---- warp-MMA validation path: fp32 activations between layers
            const float* in = xin;
            float* out = reinterpret_cast<float*>(buf0);
            for (int l = 0; l < L; ++l) {
                const LayerOff& lo = m.layers[l];
                GemmArgs g;
                g.A = in; g.lda = lo.D; g.rows_per_batch = rows; g.a_batch_stride = 0; g.M = rows;
                g.N = 2 * kGates; g.K = lo.D; g.Kp = lo.Kp;
                g.W_hi = reinterpret_cast<const __half*>(pk + lo.wih_hi);
                g.W_lo = reinterpret_cast<const __half*>(pk + lo.wih_lo);
                g.bias = reinterpret_cast<const float*>(pk + lo.bias);
                g.C = xg; g.ldc = 2 * kGates; g.c_half = 0; g.act = 0;
                if ((rc = gemm_launch(g, 0, 3, st))) return rc;
                if ((rc = lstm_recurrent_launch(xg, reinterpret_cast<const __half*>(pk + lo.whh), out, bc, (int)T, st))) return rc;
                in = out;
                out = (out == reinterpret_cast<float*>(buf0)) ? reinterpret_cast<float*>(buf1) : reinterpret_cast<float*>(buf0);
            }
            if ((rc = head_forward(m, pk, in, rows, xg, xg + rows * kHidden, prob + b0 * T, st))) return rc;
            continue;
        }
        // ---- tcgen05 path: activations travel between layers (and into the head) as fp16 (hi, lo) planes
        const __half* a_hi = x_hi;
        const __half* a_lo = x_lo;
        if (!xin) {
            a_hi = xp_hi + b0 * T * D8; a_lo = xp_lo + b0 * T * D8;                // planes straight from the front end
        } else {
            if (D % 8 == 0) rc = split_planes_launch(xin, rows * D, x_hi, x_lo, st);
            else rc = split_planes_pad_launch(xin, rows, D, D8, x_hi, x_lo, st);   // e.g. the 60 SincNet channels -> pitch 64
            if (rc) return rc;
        }
        int64_t lda = D8;
        char* outbuf = buf0;
        for (int l = 0; l < L; ++l) {
            const LayerOff& lo = m.layers[l];
            const __half* w_hi = reinterpret_cast<const __half*>(pk + lo.wih_hi);
            const __half* w_lo = reinterpret_cast<const __half*>(pk + lo.wih_lo);
            const float* bias = reinterpret_cast<const float*>(pk + lo.bias);
            // hi + lo weight planes stay resident in tensor memory: 256 k-values per launch; wider inputs (768-dim SSL
            // features on layer 0) are split along K and accumulated into xg
            int* const sync = reinterpret_cast<int*>(x_hi);
            const size_t sync_bytes = 2 * align_up(sizeof(__half) * D8 * rows);
            const int terms = (l > 0 && g_proj_terms == 2) ? 2 : 3;
            if (lstm_mode() && lstm_fused_supported(lo.D)) {
                // one kernel per layer: W_ih and W_hh (two planes each) resident in tensor memory, no xg round trip
                __half* fyh = reinterpret_cast<__half*>(outbuf);
                __half* fyl = fyh + rows * 2 * kHidden;
                const int fscaled = (g_proj_terms == 2 && l + 1 < L) ? 1 : 0;
                if (lstm_mode() == 2)
                    rc = lstm_pair_launch(a_hi, a_lo, lda, bc, (int)T, lo.D, w_hi, w_lo, lo.Kp, reinterpret_cast<const __half*>(pk + lo.whh),
                                          reinterpret_cast<const __half*>(pk + lo.whh_lo), bias, terms, fyh, fyl, st);
                else
                    rc = lstm_fused_launch(a_hi, a_lo, lda, bc, (int)T, lo.D, w_hi, w_lo, lo.Kp, reinterpret_cast<const __half*>(pk + lo.whh),
                                           reinterpret_cast<const __half*>(pk + lo.whh_lo), bias, terms, fyh, fyl, fscaled, st);
                if (rc) return rc;
                a_hi = fyh; a_lo = fyl; lda = 2 * kHidden;
                outbuf = (outbuf == buf0) ? buf1 : buf0;
                continue;
            }
            if (g_proj_kernel != 0 && lo.D <= 256) {
                // one launch, both weight planes resident in TMEM; the lockstep counters live in the layer-0 input planes'
                // workspace, which is free when the planes come from the fused fbank and dead after layer 0
                int* const sy = (l == 0 && xin) ? nullptr : sync;
                if (g_proj_kernel == 2)      // CTA pairs share every activation tile (cta_group::2 MMAs)
                    rc = gemm_xg_pair_launch(a_hi, a_lo, lda, bc, (int)T, lo.D, w_hi, w_lo, lo.Kp, lo.Kp, bias, terms, xg, sy, sync_bytes, sms, st);
                else
                    rc = gemm_xg2_launch(a_hi, a_lo, lda, bc, (int)T, lo.D, w_hi, w_lo, lo.Kp, lo.Kp, bias, terms, xg, sy, sync_bytes, sms, st);
                if (rc) return rc;
            } else
            for (int k0 = 0; k0 < lo.D; k0 += 256) {
                const int kc = std::min(256, lo.D - k0);
                if ((rc = gemm_ts_xg_launch(a_hi + k0, a_lo + k0, lda, bc, (int)T, kc, w_hi + k0, w_lo + k0, round64(kc), lo.Kp, bias,
                                            k0 > 0, xg, sms, st))) return rc;
            }
            __half* yh = reinterpret_cast<__half*>(outbuf);
            __half* yl = yh + rows * 2 * kHidden;
            // the output planes of a layer that feeds a 2-MMA projection use that kernel's scaled split; the last layer
            // (into the head's 3-term product) keeps hi / lo.  In modes 1 and 2 the next layer is a fused kernel, which
            // takes 2 products whatever g_proj_kernel says; in mode 0 kernel 0 always takes 3.
            const int scaled = (g_proj_terms == 2 && l + 1 < L && (lstm_mode() != 0 || g_proj_kernel != 0)) ? 1 : 0;
            if ((rc = lstm_tc_launch(xg, reinterpret_cast<const __half*>(pk + lo.whh), yh, yl, bc, (int)T, scaled, st))) return rc;
            a_hi = yh; a_lo = yl; lda = 2 * kHidden;
            outbuf = (outbuf == buf0) ? buf1 : buf0;
        }
        // head (PyanNet2.py:183-187) on the same GEMM: planes -> lrelu -> planes -> lrelu -> classifier -> sigmoid;
        // the classifier + sigmoid are the epilogue of the second GEMM; the z1 planes live in the xg buffer (free after
        // the last recurrence).
        if (g_head_fused) {
            if ((rc = head_fused_launch(a_hi, a_lo, rows, reinterpret_cast<const __half*>(pk + m.w1_hi),
                                        reinterpret_cast<const __half*>(pk + m.w1_lo), reinterpret_cast<const __half*>(pk + m.w2_hi),
                                        reinterpret_cast<const __half*>(pk + m.w2_lo), reinterpret_cast<const float*>(pk + m.b1),
                                        reinterpret_cast<const float*>(pk + m.b2), reinterpret_cast<const float*>(pk + m.wc),
                                        reinterpret_cast<const float*>(pk + m.bc), prob + b0 * T, sms, st))) return rc;
            continue;
        }
        __half* z1_hi = reinterpret_cast<__half*>(xg);
        __half* z1_lo = z1_hi + rows * kHidden;
        if ((rc = gemm_ts_launch(a_hi, a_lo, 2 * kHidden, rows, 2 * kHidden, reinterpret_cast<const __half*>(pk + m.w1_hi),
                                 reinterpret_cast<const __half*>(pk + m.w1_lo), 2 * kHidden, 2 * kHidden, kHidden,
                                 reinterpret_cast<const float*>(pk + m.b1), 1, 0, nullptr, z1_hi, z1_lo, kHidden, sms, st))) return rc;
        if ((rc = gemm_ts_launch(z1_hi, z1_lo, kHidden, rows, kHidden, reinterpret_cast<const __half*>(pk + m.w2_hi),
                                 reinterpret_cast<const __half*>(pk + m.w2_lo), kHidden, kHidden, kHidden,
                                 reinterpret_cast<const float*>(pk + m.b2), 4, 0, prob + b0 * T, nullptr, nullptr, 1, sms, st,
                                 reinterpret_cast<const float*>(pk + m.wc), reinterpret_cast<const float*>(pk + m.bc)))) return rc;
    }
    return B200VAD_OK;
}

// ---------------------------------------------------------------- SincNet packed layout
struct SincLayout {
    size_t filt, sinc_hi, sinc_lo, c1_f32, c1_hi, c1_lo, c1_b, c2_f32, c2_hi, c2_lo, c2_b, wn_w, wn_b, n0_w, n0_b, n1_w, n1_b,
        n2_w, n2_b, tmp_f32, sinc_t_hi, sinc_t_lo, c1_t_hi, c1_t_lo, c2_t_hi, c2_t_lo, total;
};
// tcgen05 path: weights zero padded to 128 output rows; conv2's 60 input channels are padded to 64 (16-byte rows)
constexpr int kSincTLd = 256, kC1TLd = 448, kC2Cp = 64, kC2TLd = 5 * kC2Cp;
constexpr int kSincStep = 270;   // samples between SincNet frames: 10 x 3 x 3 x 3 (receptive_field.py)
constexpr int kSincK = 251, kSincKp = 256, kC1K = 400, kC1Kp = 416, kC2K = 300, kC2Kp = 320;
static SincLayout sinc_layout() {
    SincLayout s;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes); return o; };
    s.filt = take(sizeof(float) * 80 * kSincK);
    s.sinc_hi = take(sizeof(__half) * 80 * kSincKp);
    s.sinc_lo = take(sizeof(__half) * 80 * kSincKp);
    s.c1_f32 = take(sizeof(float) * 60 * kC1K);
    s.c1_hi = take(sizeof(__half) * 60 * kC1Kp);
    s.c1_lo = take(sizeof(__half) * 60 * kC1Kp);
    s.c1_b = take(sizeof(float) * 60);
    s.c2_f32 = take(sizeof(float) * 60 * kC2K);
    s.c2_hi = take(sizeof(__half) * 60 * kC2Kp);
    s.c2_lo = take(sizeof(__half) * 60 * kC2Kp);
    s.c2_b = take(sizeof(float) * 60);
    s.wn_w = take(4); s.wn_b = take(4);
    s.n0_w = take(sizeof(float) * 80); s.n0_b = take(sizeof(float) * 80);
    s.n1_w = take(sizeof(float) * 60); s.n1_b = take(sizeof(float) * 60);
    s.n2_w = take(sizeof(float) * 60); s.n2_b = take(sizeof(float) * 60);
    s.tmp_f32 = take(sizeof(float) * 128 * kC1TLd);
    s.sinc_t_hi = take(sizeof(__half) * 128 * kSincTLd); s.sinc_t_lo = take(sizeof(__half) * 128 * kSincTLd);
    s.c1_t_hi = take(sizeof(__half) * 128 * kC1TLd); s.c1_t_lo = take(sizeof(__half) * 128 * kC1TLd);
    s.c2_t_hi = take(sizeof(__half) * 128 * kC2TLd); s.c2_t_lo = take(sizeof(__half) * 128 * kC2TLd);
    s.total = off;
    return s;
}
struct SincDims {
    int64_t L1, P1, L2, P2, L3, P3;
};
static SincDims sinc_dims(int64_t N) {
    SincDims d;
    d.L1 = N >= 251 ? (N - 251) / 10 + 1 : 0;
    d.P1 = d.L1 / 3;
    d.L2 = d.P1 >= 5 ? d.P1 - 4 : 0;
    d.P2 = d.L2 / 3;
    d.L3 = d.P2 >= 5 ? d.P2 - 4 : 0;
    d.P3 = d.L3 / 3;
    return d;
}
// B200VAD_SINC_FUSED=0 selects the unfused sinc layer (four row-class GEMMs + pooling kernel; validation): it needs the
// (B, L1, 80) convolution output in the workspace, the fused kernel does not
static bool sinc_fused() {
    static int fused = -1;
    if (fused < 0) { const char* e = getenv("B200VAD_SINC_FUSED"); fused = (e && atoi(e) == 0) ? 0 : 1; }
    return fused != 0;
}
static inline int64_t sinc_np(int64_t N) { return (N + 16 + 7) / 8 * 8; }     // padded length of a shifted waveform copy
// rows per front-end launch: the warp-MMA GEMM grid limit (65000 x 128 conv rows) and the per-row kernels' grid.y
static int64_t sinc_chunk_rows(int64_t N) {
    return std::min<int64_t>(60000, std::max<int64_t>(1, 65000LL * 128 / std::max<int64_t>(sinc_dims(N).L1, 1)));
}
static size_t sinc_ws_per_row(int64_t N) {
    SincDims d = sinc_dims(N);
    // normalised wave (fp32, or 4 shifted fp16 hi/lo copies) + conv1 out + pooled1 (+ planes) + conv2 out + pooled2 (+ planes)
    // + conv3 out, stats
    const bool conv1_out = !(sinc_fused() && g_impl == 2);
    return align_up(std::max<size_t>(sizeof(float) * N, 16 * (size_t)sinc_np(N))) + (conv1_out ? align_up(sizeof(float) * d.L1 * 80) : 0) +
           2 * align_up(sizeof(float) * d.P1 * 80) + (conv1_out ? align_up(sizeof(float) * d.L2 * 60) : 0) + align_up(sizeof(float) * d.P2 * 60) +
           align_up(sizeof(float) * d.P2 * kC2Cp) + (conv1_out ? align_up(sizeof(float) * d.L3 * 60) : 0) + align_up(sizeof(double) * 2 * 80) + 4096;
}

}  // namespace b200vad

using namespace b200vad;

extern "C" {

int b200vad_abi_version(void) { return B200VAD_ABI_VERSION; }
const char* b200vad_last_error(void) { return g_err; }

long long b200vad_launch_count(void) { return g_launches.load(); }

void b200vad_profile_enable(int on) {
    std::lock_guard<std::mutex> lk(g_prof_mu);
    g_prof_on = on != 0;
    g_prof_used = 0;      // (re)starts a collection window
}

int b200vad_profile_collect(int kind, double* total_ms, int* launches) {
    std::lock_guard<std::mutex> lk(g_prof_mu);
    double tot = 0.0;
    int n = 0;
    for (size_t i = 0; i < g_prof_used; ++i) {
        if (g_prof_events[i].kind != kind) continue;
        B200VAD_CUDA(cudaEventSynchronize(g_prof_events[i].b));
        float ms = 0.f;
        B200VAD_CUDA(cudaEventElapsedTime(&ms, g_prof_events[i].a, g_prof_events[i].b));
        tot += ms;
        ++n;
    }
    if (total_ms) *total_ms = tot;
    if (launches) *launches = n;
    return B200VAD_OK;
}

int b200vad_set_impl(int impl) {
    B200VAD_CHECK_ARG(impl == 1 || impl == 2, "impl must be 1 (warp-MMA) or 2 (tcgen05)");
#ifndef B200VAD_VALIDATE
    if (impl == 1) {
        set_error("b200vad_set_impl(1): the warp-MMA validation kernels are not in this build (make VALIDATE=1)");
        return B200VAD_ESTATE;
    }
#endif
    g_impl = impl;
    return B200VAD_OK;
}

int b200vad_set_projection_terms(int terms) {
    B200VAD_CHECK_ARG(terms == 2 || terms == 3, "terms must be 2 or 3");
    g_proj_terms = terms;
    return B200VAD_OK;
}

void* b200vad_host_alloc(size_t bytes, int write_combined) {
    void* p = nullptr;
    const unsigned flags = cudaHostAllocPortable | (write_combined ? cudaHostAllocWriteCombined : 0u);
    if (cudaHostAlloc(&p, bytes ? bytes : 1, flags) != cudaSuccess) {
        set_error("b200vad_host_alloc: cudaHostAlloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(cudaGetLastError()));
        return nullptr;
    }
    return p;
}

void b200vad_host_free(void* p) {
    if (p) cudaFreeHost(p);
}

int b200vad_set_head_fused(int on) {
    g_head_fused = on != 0;
    return B200VAD_OK;
}

int b200vad_set_projection_kernel(int which) {
    B200VAD_CHECK_ARG(which >= 0 && which <= 2, "which must be 0, 1 or 2");
    g_proj_kernel = which;
    return B200VAD_OK;
}

int b200vad_set_lstm_fused(int on) {
    B200VAD_CHECK_ARG(on >= 0 && on <= 2, "mode must be 0 (projection + recurrence kernels), 1 (fused layer kernel) or 2 (fused, CTA-pair MMAs)");
    g_lstm_fused = on;
    return B200VAD_OK;
}
int b200vad_set_lstm_pair_opt(int opt) {
    B200VAD_CHECK_ARG(opt >= 0 && opt <= 127, "opt is a bit mask: 1 input products yield to recurrent ones, 2 double-buffered h tiles; 4, 8, 32 are timing probes (wrong results)");
    lstm_pair_set_opt(opt);
    return B200VAD_OK;
}
int b200vad_lstm_fused_clusters(void) { return lstm_fused_clusters(); }
int b200vad_set_lstm_fused_debug(int flags, int lag) {
    lstm_fused_set_debug(flags, lag);
    return B200VAD_OK;
}
int b200vad_lstm_fused_last_timeout(int* out7) {
    B200VAD_CHECK_ARG(out7, "null buffer");
    int rc = lstm_fused_last_timeout(out7);
    if (rc == B200VAD_OK && out7[0] == 0) rc = lstm_pair_last_timeout(out7);
    return rc;
}
int b200vad_lstm_fused_read_debug(long long* host, int n) {
    B200VAD_CHECK_ARG(host && n != 0, "null buffer");
    if (n > 0 && lstm_mode() == 2) return lstm_pair_read_debug(host, n);
    return lstm_fused_read_debug(host, n);
}
int b200vad_set_lstm_tile(int sequences_per_cta) {
    int rc = lstm_tc_set_tile(sequences_per_cta);
    if (rc) set_error("b200vad_set_lstm_tile: must be 0 (automatic), 16 or 64");
    return rc;
}

int b200vad_init(int device) {
    int n = 0;
    B200VAD_CUDA(cudaGetDeviceCount(&n));
    B200VAD_CHECK_ARG(device >= 0 && device < n, "no such CUDA device");
    B200VAD_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    B200VAD_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        set_error("b200vad_init: device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
        return B200VAD_ESTATE;
    }
    return fbank_tables_init(device);
}

int64_t b200vad_fbank_num_frames(int64_t n) { return n < 0 ? 0 : (n + kFrameShift / 2) / kFrameShift; }

static int fbank_entry(const void* wav, int wav_i16, const int32_t* lens, int B, int64_t N, int64_t wav_stride, float* feats,
                       int64_t T, double* row_sum_ws, void* stream) {
    B200VAD_CHECK_ARG(B >= 0 && N >= 0 && T >= 0, "negative size");
    if (B == 0 || T == 0) return B200VAD_OK;
    B200VAD_CHECK_ARG(wav && feats && row_sum_ws, "null pointer");
    B200VAD_CHECK_ARG(N >= 1 && wav_stride >= 1, "need N >= 1 and wav_stride >= 1 (rows may overlap: long-form windows)");
    B200VAD_CHECK_ARG(B <= 65535, "B must be <= 65535 per call");
    int dev = 0;
    B200VAD_CUDA(cudaGetDevice(&dev));
    return fbank_launch(wav, wav_i16, lens, B, N, wav_stride, feats, nullptr, nullptr, T, row_sum_ws, dev, (cudaStream_t)stream);
}
int b200vad_fbank_f32(const float* wav, const int32_t* lens, int B, int64_t N, int64_t wav_stride, float* feats, int64_t T,
                      double* row_sum_ws, void* stream) {
    return fbank_entry(wav, 0, lens, B, N, wav_stride, feats, T, row_sum_ws, stream);
}
int b200vad_fbank_i16(const int16_t* wav, const int32_t* lens, int B, int64_t N, int64_t wav_stride, float* feats, int64_t T,
                      double* row_sum_ws, void* stream) {
    return fbank_entry(wav, 1, lens, B, N, wav_stride, feats, T, row_sum_ws, stream);
}

size_t b200vad_model_packed_bytes(int D, int L) {
    if (D <= 0 || D > B200VAD_MAX_INPUT_DIM || L <= 0) return 0;
    return model_layout(D, L).total;
}

int b200vad_model_pack_lstm(void* packed, int D, int L, int layer, int dir, const float* w_ih, const float* w_hh,
                            const float* b_ih, const float* b_hh, void* stream) {
    B200VAD_CHECK_ARG(D <= B200VAD_MAX_INPUT_DIM, "input width D > 768 (the widest supported input, B200VAD_MAX_INPUT_DIM)");
    B200VAD_CHECK_ARG(packed && w_ih && w_hh && b_ih && b_hh, "null pointer");
    B200VAD_CHECK_ARG(D > 0 && L > 0 && layer >= 0 && layer < L && (dir == 0 || dir == 1), "bad index");
    ModelLayout m = model_layout(D, L);
    const LayerOff& lo = m.layers[layer];
    char* pk = reinterpret_cast<char*>(packed);
    cudaStream_t st = (cudaStream_t)stream;
    int rc = split_weights(w_ih, kGates, lo.D, lo.Kp, reinterpret_cast<__half*>(pk + lo.wih_hi) + (size_t)dir * kGates * lo.Kp,
                           reinterpret_cast<__half*>(pk + lo.wih_lo) + (size_t)dir * kGates * lo.Kp, st, 1);
    if (rc) return rc;
    rc = add_bias(b_ih, b_hh, reinterpret_cast<float*>(pk + lo.bias) + dir * kGates, kGates, st);
    if (rc) return rc;
    return pack_whh(w_hh, reinterpret_cast<__half*>(pk + lo.whh) + (size_t)dir * kGates * kHidden, st,
                    reinterpret_cast<__half*>(pk + lo.whh_lo) + (size_t)dir * kGates * kHidden);
}

int b200vad_model_pack_head(void* packed, int D, int L, const float* w1, const float* b1, const float* w2, const float* b2,
                            const float* wc, const float* bc, void* stream) {
    B200VAD_CHECK_ARG(D <= B200VAD_MAX_INPUT_DIM, "input width D > 768 (the widest supported input, B200VAD_MAX_INPUT_DIM)");
    B200VAD_CHECK_ARG(packed && w1 && b1 && w2 && b2 && wc && bc, "null pointer");
    B200VAD_CHECK_ARG(D > 0 && L > 0, "bad shape");
    ModelLayout m = model_layout(D, L);
    char* pk = reinterpret_cast<char*>(packed);
    cudaStream_t st = (cudaStream_t)stream;
    int rc = split_weights(w1, kHidden, 2 * kHidden, 2 * kHidden, reinterpret_cast<__half*>(pk + m.w1_hi),
                           reinterpret_cast<__half*>(pk + m.w1_lo), st);
    if (rc) return rc;
    rc = split_weights(w2, kHidden, kHidden, kHidden, reinterpret_cast<__half*>(pk + m.w2_hi),
                       reinterpret_cast<__half*>(pk + m.w2_lo), st);
    if (rc) return rc;
    B200VAD_CUDA(cudaMemcpyAsync(pk + m.b1, b1, sizeof(float) * kHidden, cudaMemcpyDeviceToDevice, st));
    B200VAD_CUDA(cudaMemcpyAsync(pk + m.b2, b2, sizeof(float) * kHidden, cudaMemcpyDeviceToDevice, st));
    B200VAD_CUDA(cudaMemcpyAsync(pk + m.wc, wc, sizeof(float) * kHidden, cudaMemcpyDeviceToDevice, st));
    B200VAD_CUDA(cudaMemcpyAsync(pk + m.bc, bc, sizeof(float), cudaMemcpyDeviceToDevice, st));
    return B200VAD_OK;
}

size_t b200vad_model_workspace_bytes(int B, int64_t T) {
    if (B <= 0 || T <= 0) return 0;
    return (size_t)ceil64(B) * model_per_row(B200VAD_MAX_INPUT_DIM, T) + 4096;   /* whole 64-sequence blocks, widest supported input */
}

int b200vad_model_forward_f32(const void* packed, int D, int L, const float* x, int B, int64_t T, float* prob, void* ws,
                              size_t ws_bytes, void* stream) {
    return model_forward(packed, D, L, x, nullptr, nullptr, B, T, prob, ws, ws_bytes, (cudaStream_t)stream);
}

int b200vad_linear_split_f32(const float* a, int64_t M, int K, const float* w, int N, const float* bias, int use_w_lo, float* c,
                             void* ws, size_t ws_bytes, void* stream) {
    B200VAD_CHECK_ARG(a && w && c && ws, "null pointer");
    B200VAD_CHECK_ARG(M >= 0 && K > 0 && K % 8 == 0 && N > 0 && N % 128 == 0, "need K % 8 == 0 and N % 128 == 0");
    B200VAD_CHECK_ARG((use_w_lo ? 2 : 1) * round64(K) <= 512, "weights must fit in tensor memory: planes x K <= 512");
    B200VAD_CHECK_ARG((reinterpret_cast<uintptr_t>(ws) & 255) == 0, "workspace must be 256-byte aligned");
    const int Kp = round64(K);
    const size_t need = 2 * align_up(sizeof(__half) * M * K) + 2 * align_up(sizeof(__half) * (size_t)N * Kp);
    if (ws_bytes < need) {
        set_error("linear_split: workspace too small (%zu < %zu)", ws_bytes, need);
        return B200VAD_ENOMEM;
    }
    cudaStream_t st = (cudaStream_t)stream;
    char* p = reinterpret_cast<char*>(ws);
    __half* a_hi = reinterpret_cast<__half*>(p); p += align_up(sizeof(__half) * M * K);
    __half* a_lo = reinterpret_cast<__half*>(p); p += align_up(sizeof(__half) * M * K);
    __half* w_hi = reinterpret_cast<__half*>(p); p += align_up(sizeof(__half) * (size_t)N * Kp);
    __half* w_lo = reinterpret_cast<__half*>(p);
    int rc = split_planes_launch(a, M * K, a_hi, a_lo, st);
    if (rc) return rc;
    if ((rc = split_weights(w, N, K, Kp, w_hi, w_lo, st))) return rc;
    return gemm_ts_launch(a_hi, a_lo, K, M, K, w_hi, use_w_lo ? w_lo : nullptr, Kp, Kp, N, bias, 0, 0, c, nullptr, nullptr, N,
                          num_sms_cached(), st);
}

// ---------------------------------------------------------------- SincNet
int64_t b200vad_sincnet_num_frames(int64_t n) { return sinc_dims(n).P3; }
size_t b200vad_sincnet_packed_bytes(void) { return sinc_layout().total; }

int b200vad_sincnet_pack(void* packed, const float* wav_norm_w, const float* wav_norm_b, const float* low_hz,
                         const float* band_hz, const float* window, const float* n, const float* conv1_w,
                         const float* conv1_b, const float* conv2_w, const float* conv2_b, const float* norm0_w,
                         const float* norm0_b, const float* norm1_w, const float* norm1_b, const float* norm2_w,
                         const float* norm2_b, void* stream) {
    B200VAD_CHECK_ARG(packed && wav_norm_w && wav_norm_b && low_hz && band_hz && window && n && conv1_w && conv1_b &&
                          conv2_w && conv2_b && norm0_w && norm0_b && norm1_w && norm1_b && norm2_w && norm2_b,
                      "null pointer");
    SincLayout s = sinc_layout();
    char* pk = reinterpret_cast<char*>(packed);
    cudaStream_t st = (cudaStream_t)stream;
    int rc = sinc_filters_launch(low_hz, band_hz, window, n, reinterpret_cast<float*>(pk + s.filt), st);
    if (rc) return rc;
    rc = split_weights(reinterpret_cast<float*>(pk + s.filt), 80, kSincK, kSincKp, reinterpret_cast<__half*>(pk + s.sinc_hi),
                       reinterpret_cast<__half*>(pk + s.sinc_lo), st);
    if (rc) return rc;
    rc = repack_conv_launch(conv1_w, 60, 80, 5, reinterpret_cast<float*>(pk + s.c1_f32), st);
    if (rc) return rc;
    rc = split_weights(reinterpret_cast<float*>(pk + s.c1_f32), 60, kC1K, kC1Kp, reinterpret_cast<__half*>(pk + s.c1_hi),
                       reinterpret_cast<__half*>(pk + s.c1_lo), st);
    if (rc) return rc;
    rc = repack_conv_launch(conv2_w, 60, 60, 5, reinterpret_cast<float*>(pk + s.c2_f32), st);
    if (rc) return rc;
    rc = split_weights(reinterpret_cast<float*>(pk + s.c2_f32), 60, kC2K, kC2Kp, reinterpret_cast<__half*>(pk + s.c2_hi),
                       reinterpret_cast<__half*>(pk + s.c2_lo), st);
    if (rc) return rc;
    // tcgen05 path: (128, ld) zero-padded copies
    float* tmp = reinterpret_cast<float*>(pk + s.tmp_f32);
    if ((rc = pad_rows_launch(reinterpret_cast<float*>(pk + s.filt), 80, kSincK, kSincTLd, tmp, st))) return rc;
    if ((rc = split_weights(tmp, 128, kSincTLd, kSincTLd, reinterpret_cast<__half*>(pk + s.sinc_t_hi),
                            reinterpret_cast<__half*>(pk + s.sinc_t_lo), st))) return rc;
    if ((rc = repack_conv_pad_launch(conv1_w, 60, 80, 5, 80, kC1TLd, tmp, st))) return rc;
    if ((rc = split_weights(tmp, 128, kC1TLd, kC1TLd, reinterpret_cast<__half*>(pk + s.c1_t_hi),
                            reinterpret_cast<__half*>(pk + s.c1_t_lo), st))) return rc;
    if ((rc = repack_conv_pad_launch(conv2_w, 60, 60, 5, kC2Cp, kC2TLd, tmp, st))) return rc;
    if ((rc = split_weights(tmp, 128, kC2TLd, kC2TLd, reinterpret_cast<__half*>(pk + s.c2_t_hi),
                            reinterpret_cast<__half*>(pk + s.c2_t_lo), st))) return rc;
    struct { size_t off; const float* src; size_t n; } cp[] = {
        {s.c1_b, conv1_b, 60}, {s.c2_b, conv2_b, 60}, {s.wn_w, wav_norm_w, 1}, {s.wn_b, wav_norm_b, 1},
        {s.n0_w, norm0_w, 80}, {s.n0_b, norm0_b, 80}, {s.n1_w, norm1_w, 60}, {s.n1_b, norm1_b, 60},
        {s.n2_w, norm2_w, 60}, {s.n2_b, norm2_b, 60}};
    for (auto& c : cp) B200VAD_CUDA(cudaMemcpyAsync(pk + c.off, c.src, sizeof(float) * c.n, cudaMemcpyDeviceToDevice, st));
    return B200VAD_OK;
}

size_t b200vad_sincnet_workspace_bytes(int B, int64_t N) {
    if (B <= 0 || N <= 0) return 0;
    return (size_t)B * sinc_ws_per_row(N) + 4096;
}

// SincNet front end on (B, N) rows `wav_stride` samples apart (f32, or int16 PCM with wav_i16), in chunks of rows that fit
// the workspace.  Output: `out` (B, Ts, 60) f32, or -- tcgen05 path, o_hi / o_lo given -- the LSTM's layer-0 operand as fp16
// (hi, lo) planes (B, Ts, 64) with channels 60..63 zero: the unscaled split of split_planes_pad_kernel, so model_forward sees
// the same bits either way, without the fp32 round trip through HBM and the split pass.  Every chunk writes its own rows of
// the whole-batch output.
// rows != nullptr (tcgen05 path only): row b starts at rows[b] and has lens[b] valid samples, the rest read as 0 (wav is unused).
static int sincnet_forward(const void* packed, const void* wav, int wav_i16, int B, int64_t N, int64_t wav_stride, float* out,
                           __half* o_hi, __half* o_lo, void* workspace, size_t ws_bytes, cudaStream_t st,
                           const void* const* rows = nullptr, const int32_t* lens = nullptr) {
    const bool planes = o_hi != nullptr;
    B200VAD_CHECK_ARG(packed && (wav || (rows && lens)) && (out || (o_hi && o_lo)) && workspace, "null pointer");
    B200VAD_CHECK_ARG(B >= 0 && N >= 0 && wav_stride >= 1, "bad shape");
    B200VAD_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "workspace must be 256-byte aligned");
    const SincDims d = sinc_dims(N);
    B200VAD_CHECK_ARG(d.P3 >= 1, "waveform shorter than the SincNet receptive field (991 samples)");
    if ((planes || wav_i16 || rows) && g_impl != 2) {
        set_error("sincnet: int16 input, row tables and plane output need the tcgen05 path (b200vad_set_impl(2))");
        return B200VAD_ESTATE;
    }
    if (B == 0) return B200VAD_OK;
    const SincLayout s = sinc_layout();
    const char* pk = reinterpret_cast<const char*>(packed);
    const size_t per_row = sinc_ws_per_row(N);
    int64_t Bc = std::min<int64_t>((int64_t)(ws_bytes / per_row), B);
    Bc = std::min<int64_t>(Bc, sinc_chunk_rows(N));
    if (Bc < 1) {
        set_error("sincnet_forward: workspace too small (%zu bytes; need >= %zu per row)", ws_bytes, per_row);
        return B200VAD_ENOMEM;
    }
    for (int64_t b0 = 0; b0 < B; b0 += Bc) {
        const int bc = (int)std::min<int64_t>(Bc, B - b0);
        char* w = reinterpret_cast<char*>(workspace);
        auto take = [&](size_t bytes) { char* p = w; w += align_up(bytes); return p; };
        const int64_t Np = sinc_np(N);
        char* wn_raw = take(std::max<size_t>(sizeof(float) * N, 16 * (size_t)Np) * bc);
        float* wn = reinterpret_cast<float*>(wn_raw);
        float* c1 = (sinc_fused() && g_impl == 2) ? nullptr : reinterpret_cast<float*>(take(sizeof(float) * d.L1 * 80 * bc));
        float* p1 = reinterpret_cast<float*>(take(sizeof(float) * d.P1 * 80 * bc));
        __half* p1_hi = reinterpret_cast<__half*>(take(sizeof(float) * d.P1 * 80 * bc));
        __half* p1_lo = p1_hi + d.P1 * 80 * bc;
        const bool fused_convs = sinc_fused() && g_impl == 2;
        float* c2 = fused_convs ? nullptr : reinterpret_cast<float*>(take(sizeof(float) * d.L2 * 60 * bc));
        float* p2 = reinterpret_cast<float*>(take(sizeof(float) * d.P2 * 60 * bc));
        __half* p2_hi = reinterpret_cast<__half*>(take(sizeof(float) * d.P2 * kC2Cp * bc));
        __half* p2_lo = p2_hi + d.P2 * kC2Cp * bc;
        float* c3 = fused_convs ? nullptr : reinterpret_cast<float*>(take(sizeof(float) * d.L3 * 60 * bc));
        double* stats = reinterpret_cast<double*>(take(sizeof(double) * 2 * 80 * bc));
        __half* const o3_hi = planes ? o_hi + b0 * d.P3 * kC2Cp : nullptr;
        __half* const o3_lo = planes ? o_lo + b0 * d.P3 * kC2Cp : nullptr;
        int rc;
        if (g_impl == 2) {
            // ---- tcgen05 path: every convolution is an overlapping-row GEMM on gemm_ts (weights resident in TMEM)
            const int sms = num_sms_cached();
            __half* wn_hi = reinterpret_cast<__half*>(wn_raw);
            __half* wn_lo = wn_hi + 4 * (int64_t)bc * Np;
            const void* wrow = rows ? nullptr : reinterpret_cast<const char*>(wav) + (wav_i16 ? sizeof(int16_t) : sizeof(float)) * b0 * wav_stride;
            if ((rc = wave_norm_planes_launch(wrow, wav_i16, bc, N, wav_stride, Np, reinterpret_cast<const float*>(pk + s.wn_w),
                                              reinterpret_cast<const float*>(pk + s.wn_b), stats, wn_hi, wn_lo, st, 0,
                                              rows ? rows + b0 : nullptr, rows ? lens + b0 : nullptr))) return rc;
            if (sinc_fused()) {
                // (three fp16 products per k-step: the 2-product scheme of the LSTM projections costs 3e-3 on the normalised SincNet
            // output -- three convolutions and InstanceNorms amplify it -- for 4 % of the front-end time; the kernels keep the option)
            // sinc conv + |x| + MaxPool3 + InstanceNorm sums in one launch: the (B, L1, 80) convolution output never exists
                if ((rc = zero_f64_launch(stats, (int64_t)2 * bc * 80, st))) return rc;
                if ((rc = sinc_pool_gemm_launch(wn_hi, wn_lo, Np, bc, d.L1, reinterpret_cast<const __half*>(pk + s.sinc_t_hi),
                                                reinterpret_cast<const __half*>(pk + s.sinc_t_lo), kSincTLd, kSincTLd, 80, 3, p1, 80, stats,
                                                sms, st))) return rc;
                if ((rc = norm_lrelu_launch(p1, bc, d.P1, 80, stats, reinterpret_cast<const float*>(pk + s.n0_w),
                                            reinterpret_cast<const float*>(pk + s.n0_b), st, p1_hi, p1_lo, 80, 0))) return rc;
            } else {
            // sinc conv, stride 10: rows t = 4 m + r start at 40 m + 10 r -> copy shifted by (10 r) % 8, offset 8 * ((10 r) / 8)
                for (int r = 0; r < 4; ++r) {
                    const int64_t rows_r = (d.L1 - r + 3) / 4;
                    if (rows_r <= 0) continue;
                    const int e = ((10 * r) % 8) / 2, q = ((10 * r) / 8) * 8;
                    if ((rc = gemm_ts_rows_launch(wn_hi + (int64_t)e * bc * Np + q, wn_lo + (int64_t)e * bc * Np + q, 40, Np, bc, (int)rows_r,
                                                  kSincTLd, reinterpret_cast<const __half*>(pk + s.sinc_t_hi),
                                                  reinterpret_cast<const __half*>(pk + s.sinc_t_lo), kSincTLd, kSincTLd, 80, nullptr, 0, 1,
                                                  c1, 80, d.L1, 4, r, sms, st))) return rc;
                }
                if ((rc = pool_norm_lrelu_launch(c1, bc, d.L1, 80, p1, stats, reinterpret_cast<const float*>(pk + s.n0_w),
                                                 reinterpret_cast<const float*>(pk + s.n0_b), st, p1_hi, p1_lo, 80))) return rc;
            }
            const __half* w1h = reinterpret_cast<const __half*>(pk + s.c1_t_hi);
            const __half* w1l = reinterpret_cast<const __half*>(pk + s.c1_t_lo);
            const float* b1 = reinterpret_cast<const float*>(pk + s.c1_b);
            const __half* w2h = reinterpret_cast<const __half*>(pk + s.c2_t_hi);
            const __half* w2l = reinterpret_cast<const __half*>(pk + s.c2_t_lo);
            const float* b2 = reinterpret_cast<const float*>(pk + s.c2_b);
            if (sinc_fused()) {
                // Conv1d(80, 60, 5) / Conv1d(60 -> 64 padded, 60, 5): whole K resident in TMEM, bias + MaxPool3 + InstanceNorm sums
                // in the epilogue (conv_pool_gemm_kernel): neither the convolution outputs nor a K-split partial sum exist
                if ((rc = zero_f64_launch(stats, (int64_t)2 * bc * 60, st))) return rc;
                if ((rc = conv_pool_gemm_launch(p1_hi, p1_lo, 80, d.P1 * 80, bc, d.L2, kC1K, w1h, w1l, kC1TLd, kC1TLd, 60, b1, 3, p2, 60, stats,
                                                sms, st))) return rc;
                if ((rc = norm_lrelu_launch(p2, bc, d.P2, 60, stats, reinterpret_cast<const float*>(pk + s.n1_w),
                                            reinterpret_cast<const float*>(pk + s.n1_b), st, p2_hi, p2_lo, kC2Cp, 0))) return rc;
                float* o3 = planes ? p2 : out + b0 * d.P3 * 60;     // plane output: the dead pooled2 buffer takes the fp32 values
                if ((rc = zero_f64_launch(stats, (int64_t)2 * bc * 60, st))) return rc;
                if ((rc = conv_pool_gemm_launch(p2_hi, p2_lo, kC2Cp, d.P2 * kC2Cp, bc, d.L3, kC2TLd, w2h, w2l, kC2TLd, kC2TLd, 60, b2, 3, o3, 60,
                                                stats, sms, st))) return rc;
                if ((rc = norm_lrelu_launch(o3, bc, d.P3, 60, stats, reinterpret_cast<const float*>(pk + s.n2_w),
                                            reinterpret_cast<const float*>(pk + s.n2_b), st, o3_hi, o3_lo, kC2Cp, 0))) return rc;
                continue;
            }
            // Conv1d(80, 60, 5): row t = p1[b, t : t + 5, :] = 400 contiguous values, K split 256 + 144
            if ((rc = gemm_ts_rows_launch(p1_hi, p1_lo, 80, d.P1 * 80, bc, (int)d.L2, 256, w1h, w1l, 256, kC1TLd, 60, b1, 0, 0, c2, 60,
                                          d.L2, 1, 0, sms, st))) return rc;
            if ((rc = gemm_ts_rows_launch(p1_hi + 256, p1_lo + 256, 80, d.P1 * 80, bc, (int)d.L2, 144, w1h + 256, w1l + 256, 192, kC1TLd,
                                          60, nullptr, 1, 0, c2, 60, d.L2, 1, 0, sms, st))) return rc;
            if ((rc = pool_norm_lrelu_launch(c2, bc, d.L2, 60, p2, stats, reinterpret_cast<const float*>(pk + s.n1_w),
                                             reinterpret_cast<const float*>(pk + s.n1_b), st, p2_hi, p2_lo, kC2Cp))) return rc;
            // Conv1d(60, 60, 5) on channels padded to 64: row t = 320 contiguous values, K split 256 + 64
            if ((rc = gemm_ts_rows_launch(p2_hi, p2_lo, kC2Cp, d.P2 * kC2Cp, bc, (int)d.L3, 256, w2h, w2l, 256, kC2TLd, 60, b2, 0, 0, c3,
                                          60, d.L3, 1, 0, sms, st))) return rc;
            if ((rc = gemm_ts_rows_launch(p2_hi + 256, p2_lo + 256, kC2Cp, d.P2 * kC2Cp, bc, (int)d.L3, 64, w2h + 256, w2l + 256, 64,
                                          kC2TLd, 60, nullptr, 1, 0, c3, 60, d.L3, 1, 0, sms, st))) return rc;
            if ((rc = pool_norm_lrelu_launch(c3, bc, d.L3, 60, planes ? p2 : out + b0 * d.P3 * 60, stats,
                                             reinterpret_cast<const float*>(pk + s.n2_w), reinterpret_cast<const float*>(pk + s.n2_b), st,
                                             o3_hi, o3_lo, kC2Cp))) return rc;
            continue;
        }
        // ---- warp-MMA validation path
        rc = wave_instnorm_launch(reinterpret_cast<const float*>(wav) + b0 * wav_stride, bc, N, wav_stride, reinterpret_cast<const float*>(pk + s.wn_w),
                                  reinterpret_cast<const float*>(pk + s.wn_b), stats, wn, st);
        if (rc) return rc;
        GemmArgs g;
        // sinc conv: rows (b, t) = wn[b, 10 t : 10 t + 251]
        g.A = wn; g.lda = 10; g.rows_per_batch = d.L1; g.a_batch_stride = N; g.M = d.L1 * bc;
        g.N = 80; g.K = kSincK; g.Kp = kSincKp;
        g.W_hi = reinterpret_cast<const __half*>(pk + s.sinc_hi); g.W_lo = reinterpret_cast<const __half*>(pk + s.sinc_lo);
        g.bias = nullptr; g.C = c1; g.ldc = 80; g.c_half = 0; g.act = 2;
        rc = gemm_launch(g, 0, 3, st);
        if (rc) return rc;
        rc = pool_norm_lrelu_launch(c1, bc, d.L1, 80, p1, stats, reinterpret_cast<const float*>(pk + s.n0_w),
                                    reinterpret_cast<const float*>(pk + s.n0_b), st);
        if (rc) return rc;
        // Conv1d(80, 60, 5): rows (b, t) = p1[b, t : t + 5, :]
        g.A = p1; g.lda = 80; g.rows_per_batch = d.L2; g.a_batch_stride = d.P1 * 80; g.M = d.L2 * bc;
        g.N = 60; g.K = kC1K; g.Kp = kC1Kp;
        g.W_hi = reinterpret_cast<const __half*>(pk + s.c1_hi); g.W_lo = reinterpret_cast<const __half*>(pk + s.c1_lo);
        g.bias = reinterpret_cast<const float*>(pk + s.c1_b); g.C = c2; g.ldc = 60; g.act = 0;
        rc = gemm_launch(g, 0, 3, st);
        if (rc) return rc;
        rc = pool_norm_lrelu_launch(c2, bc, d.L2, 60, p2, stats, reinterpret_cast<const float*>(pk + s.n1_w),
                                    reinterpret_cast<const float*>(pk + s.n1_b), st);
        if (rc) return rc;
        g.A = p2; g.lda = 60; g.rows_per_batch = d.L3; g.a_batch_stride = d.P2 * 60; g.M = d.L3 * bc;
        g.N = 60; g.K = kC2K; g.Kp = kC2Kp;
        g.W_hi = reinterpret_cast<const __half*>(pk + s.c2_hi); g.W_lo = reinterpret_cast<const __half*>(pk + s.c2_lo);
        g.bias = reinterpret_cast<const float*>(pk + s.c2_b); g.C = c3; g.ldc = 60; g.act = 0;
        rc = gemm_launch(g, 0, 3, st);
        if (rc) return rc;
        rc = pool_norm_lrelu_launch(c3, bc, d.L3, 60, out + b0 * d.P3 * 60, stats, reinterpret_cast<const float*>(pk + s.n2_w),
                                    reinterpret_cast<const float*>(pk + s.n2_b), st);
        if (rc) return rc;
    }
    return B200VAD_OK;
}

int b200vad_sincnet_forward_f32(const void* packed, const float* wav, int B, int64_t N, int64_t wav_stride, float* out,
                                void* workspace, size_t ws_bytes, void* stream) {
    B200VAD_CHECK_ARG(wav_stride >= N, "bad shape");
    return sincnet_forward(packed, wav, 0, B, N, wav_stride, out, nullptr, nullptr, workspace, ws_bytes, (cudaStream_t)stream);
}

// ---------------------------------------------------------------- post-processing
int b200vad_median_window(double speech_window, double window) {
    int k = (int)(speech_window / window);   // helper.py:85-87
    if (k % 2 == 0) k -= 1;
    return k;
}

int b200vad_threshold_median(const float* prob, int B, int64_t T, float thr, int kernel, void* out, int elem_bytes,
                             int32_t* near_count, float near_tol, void* stream) {
    B200VAD_CHECK_ARG(B >= 0 && T >= 0, "negative size");
    if (B == 0 || T == 0) return B200VAD_OK;
    B200VAD_CHECK_ARG(prob && out, "null pointer");
    B200VAD_CHECK_ARG(elem_bytes == 1 || elem_bytes == 8, "elem_bytes must be 1 or 8");
    B200VAD_CHECK_ARG(B <= 65535, "B must be <= 65535 per call");
    return threshold_median_launch(prob, B, T, thr, kernel, out, elem_bytes, near_count, near_tol, (cudaStream_t)stream);
}

int b200vad_threshold_median_streams(const float* prob, const int64_t* offsets, int R, int64_t max_len, float thr, int kernel,
                                     uint8_t* out, void* stream) {
    B200VAD_CHECK_ARG(R >= 0 && R <= 65535 && max_len >= 0, "need 0 <= R <= 65535 and max_len >= 0");
    if (R == 0 || max_len == 0) return B200VAD_OK;
    B200VAD_CHECK_ARG(prob && offsets && out, "null pointer");
    return threshold_median_launch(prob, R, max_len, thr, kernel, out, 1, nullptr, 0.f, (cudaStream_t)stream, offsets);
}

// B200VAD_EINVAL unless the thresholds are finite with offset <= onset and every count is >= 0
static int check_binarize(const b200vad_binarize_params* p) {
    B200VAD_CHECK_ARG(p, "null binarize params");
    B200VAD_CHECK_ARG(std::isfinite(p->onset) && std::isfinite(p->offset) && p->offset <= p->onset,
                      "binarize: onset and offset must be finite with offset <= onset");
    B200VAD_CHECK_ARG(p->pad_onset >= 0 && p->pad_offset >= 0 && p->min_off >= 0 && p->min_on >= 0,
                      "binarize: pads and minimum durations must be >= 0 frames");
    return B200VAD_OK;
}

int b200vad_binarize(const float* prob, const int64_t* offsets, int R, int64_t T, const b200vad_binarize_params* params,
                     uint8_t* dec, int32_t* counts, int64_t* seg_off, int32_t* seg, int64_t cap, void* stream) {
    int rc = check_binarize(params);
    if (rc) return rc;
    B200VAD_CHECK_ARG(R >= 0 && T >= 0 && cap >= 0, "bad size");
    B200VAD_CHECK_ARG(offsets || T <= INT32_MAX, "T must fit the int32 frame indices of the triples");
    if (R == 0) return B200VAD_OK;
    B200VAD_CHECK_ARG(prob && dec && counts && seg_off && (seg || cap == 0), "null pointer");
    return binarize_launch(prob, offsets, T, R, *params, 0, dec, counts, seg_off, seg, cap, (cudaStream_t)stream);
}

int b200vad_regions_step(const float* prob, int S, int nf, int64_t row_stride, const b200vad_binarize_params* params,
                         int64_t* state, const uint8_t* flush, int64_t* ev, int32_t* ev_counts, int64_t cap_per_stream,
                         void* stream) {
    int rc = check_binarize(params);
    if (rc) return rc;
    B200VAD_CHECK_ARG(S >= 0 && nf >= 0 && row_stride >= nf && cap_per_stream >= 0, "bad size");
    if (S == 0) return B200VAD_OK;
    B200VAD_CHECK_ARG(state && ev_counts && (prob || nf == 0) && (ev || cap_per_stream == 0), "null pointer");
    return regions_step_launch(prob, S, nf, row_stride, *params, state, flush, ev, ev_counts, cap_per_stream, (cudaStream_t)stream);
}

int b200vad_segments(const uint8_t* dec, const int64_t* offsets, int R, int64_t T, int min_run, int32_t* counts,
                     int64_t* seg_off, int32_t* seg, int64_t cap, void* stream) {
    B200VAD_CHECK_ARG(R >= 0 && cap >= 0 && min_run >= 1, "bad size");
    if (R == 0) return B200VAD_OK;
    B200VAD_CHECK_ARG(dec && counts && seg_off && (seg || cap == 0), "null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    B200VAD_CHECK_ARG(offsets || T >= 0, "bad T");
    return segments_launch(dec, offsets, T, R, min_run, 0, counts, seg_off, seg, cap, st);
}

// ---------------------------------------------------------------- scoring (SURVEY 8f rank 1)
int b200vad_stat_scores(const uint8_t* dec, const uint8_t* labels, int64_t n, int64_t* out4, void* stream) {
    B200VAD_CHECK_ARG(n >= 0 && out4 && ((dec && labels) || n == 0), "bad argument");
    return stat_scores_launch(dec, labels, n, out4, (cudaStream_t)stream);
}

size_t b200vad_score_workspace_bytes(int64_t total_words) { return total_words <= 0 ? 256 : (size_t)total_words * 8 + 256; }

int b200vad_score_intervals(const int32_t* gt_iv, int64_t n_gt, const int32_t* pred_iv, int64_t n_pred, const int64_t* word_off,
                            const int32_t* nframes, int R, int64_t total_words, int max_words_per_rec, void* workspace,
                            int64_t* fa, int64_t* md, void* stream) {
    B200VAD_CHECK_ARG(R >= 0 && n_gt >= 0 && n_pred >= 0 && total_words >= 0, "negative size");
    if (R == 0) return B200VAD_OK;
    B200VAD_CHECK_ARG(word_off && nframes && workspace && fa && md, "null pointer");
    B200VAD_CHECK_ARG((gt_iv || n_gt == 0) && (pred_iv || n_pred == 0), "null interval list");
    B200VAD_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 15) == 0, "workspace must be 16-byte aligned");
    return score_intervals_launch(gt_iv, n_gt, pred_iv, n_pred, word_off, nframes, R, total_words,
                                  reinterpret_cast<uint32_t*>(workspace), fa, md, max_words_per_rec, (cudaStream_t)stream);
}

// ---------------------------------------------------------------- synthetic corpus (BASELINE config 4)
int b200vad_synth_corpus(float* wav, int64_t first_utt, int rows, int64_t N, uint64_t seed, void* stream) {
    B200VAD_CHECK_ARG(rows >= 0 && rows <= 65535 && N >= 0 && first_utt >= 0, "bad shape");
    B200VAD_CHECK_ARG(wav || rows == 0 || N == 0, "null pointer");
    return synth_corpus_launch(wav, first_utt, rows, N, seed, (cudaStream_t)stream);
}

// ---------------------------------------------------------------- long-form stitching (BASELINE config 3)
int b200vad_stitch_center(const float* prob, int num_windows, int frames_per_window, int hop_frames, float* out, int64_t L,
                          void* stream) {
    B200VAD_CHECK_ARG(num_windows >= 1 && frames_per_window >= 1 && hop_frames >= 1 && hop_frames <= frames_per_window && L >= 0,
                      "need 1 <= hop_frames <= frames_per_window");
    B200VAD_CHECK_ARG(prob && (out || L == 0), "null pointer");
    return stitch_center_launch(prob, nullptr, nullptr, 1, num_windows, frames_per_window, hop_frames, out, L, 4, (cudaStream_t)stream);
}

int b200vad_stitch_center_streams(const void* prob, int elem_bytes, const int64_t* win_off, const int64_t* frame_off, int R,
                                  int frames_per_window, int hop_frames, int64_t max_len, void* out, void* stream) {
    B200VAD_CHECK_ARG(elem_bytes == 1 || elem_bytes == 4, "elem_bytes must be 1 or 4");
    B200VAD_CHECK_ARG(R >= 0 && R <= 65535 && max_len >= 0, "need 0 <= R <= 65535 and max_len >= 0");
    B200VAD_CHECK_ARG(frames_per_window >= 1 && hop_frames >= 1 && hop_frames <= frames_per_window,
                      "need 1 <= hop_frames <= frames_per_window");
    if (R == 0 || max_len == 0) return B200VAD_OK;
    B200VAD_CHECK_ARG(win_off && frame_off && out, "null pointer");
    return stitch_center_launch(prob, win_off, frame_off, R, 0, frames_per_window, hop_frames, out, max_len, elem_bytes,
                                (cudaStream_t)stream);
}

// ---------------------------------------------------------------- fused device pipeline
// Front end of the whole path: the fused fbank (sinc == nullptr: a1 -> PyanNet2) or SincNet with its packed blob (a3/a4 ->
// PyanNet).  Both hand the LSTM its layer-0 operand as fp16 (hi, lo) planes with row pitch round8(D).
static inline int64_t fe_frames(bool sinc, int64_t N) { return sinc ? sinc_dims(N).P3 : b200vad_fbank_num_frames(N); }
static inline int fe_dim(bool sinc) { return sinc ? 60 : kNumMel; }
// layout: layer-0 input (fp32 features or planes, the same bytes) | fbank row sums | model workspace; the SincNet front end's
// workspace shares the model's region (it is dead before the model runs on the same stream)
static size_t fe_feat_bytes(bool sinc, int B, int64_t T) { return align_up(sizeof(float) * (size_t)B * T * round8(fe_dim(sinc))); }
static size_t fe_sums_bytes(bool sinc, int B) { return sinc ? 0 : align_up(sizeof(double) * B); }
static size_t pipeline_ws_bytes(int B, int64_t N, bool sinc = false) {
    const int64_t T = fe_frames(sinc, N);
    size_t rest = b200vad_model_workspace_bytes(B, T);
    if (sinc) rest = std::max(rest, (size_t)std::min<int64_t>(B, sinc_chunk_rows(N)) * sinc_ws_per_row(N) + 4096);
    return fe_feat_bytes(sinc, B, T) + fe_sums_bytes(sinc, B) + rest + 4096;
}
size_t b200vad_pipeline_workspace_bytes(int B, int64_t N) {
    if (B <= 0 || N <= 0) return 0;
    return pipeline_ws_bytes(B, N);
}
size_t b200vad_pipeline_sincnet_workspace_bytes(int B, int64_t N) {
    if (B <= 0 || N < 991) return 0;
    return pipeline_ws_bytes(B, N, true);
}

// rows != nullptr: row b is read from rows[b] (lens required) instead of wav + b * stride
static int pipeline_run(const void* packed, const void* sinc, int L, const void* wav, int wav_i16, const int32_t* lens, int B,
                        int64_t N, int64_t stride, float thr, int kernel, const b200vad_binarize_params* bin, int row_base, float* prob,
                        uint8_t* dec, int32_t* counts, int64_t* seg_off, int32_t* seg, int64_t cap, void* ws, size_t ws_bytes,
                        cudaStream_t st, const void* const* rows = nullptr) {
    B200VAD_CHECK_ARG(packed && (wav || (rows && lens)) && prob && dec && counts && seg_off && ws, "null pointer");
    B200VAD_CHECK_ARG((reinterpret_cast<uintptr_t>(ws) & 255) == 0, "workspace must be 256-byte aligned");
    const int64_t T = fe_frames(sinc != nullptr, N);
    const int D = fe_dim(sinc != nullptr);
    if (B == 0 || T == 0) return B200VAD_OK;
    char* w = reinterpret_cast<char*>(ws);
    float* feats = reinterpret_cast<float*>(w); w += fe_feat_bytes(sinc != nullptr, B, T);
    double* sums = reinterpret_cast<double*>(w); w += fe_sums_bytes(sinc != nullptr, B);
    size_t used = (size_t)(w - reinterpret_cast<char*>(ws));
    const size_t rest_min = sinc ? std::max(b200vad_model_workspace_bytes(1, T), sinc_ws_per_row(N)) : b200vad_model_workspace_bytes(1, T);
    if (ws_bytes < used + rest_min) {
        set_error("pipeline: workspace too small (%zu bytes)", ws_bytes);
        return B200VAD_ENOMEM;
    }
    // the tcgen05 path takes the layer-0 input as fp16 (hi, lo) planes straight from the front end (same bytes as fp32)
    __half* f_hi = reinterpret_cast<__half*>(feats);
    __half* f_lo = f_hi + (size_t)B * T * round8(D);
    const bool planes = g_impl == 2;
    int rc;
    if (sinc) {
        if (!planes) {
            set_error("pipeline: the SincNet front end runs on the tcgen05 path only (b200vad_set_impl(2))");
            return B200VAD_ESTATE;
        }
        rc = sincnet_forward(sinc, wav, wav_i16, B, N, stride, nullptr, f_hi, f_lo, w, ws_bytes - used, st, rows, lens);
    } else {
        int dev = 0;
        B200VAD_CUDA(cudaGetDevice(&dev));
        rc = fbank_launch(wav, wav_i16, lens, B, N, stride, planes ? nullptr : feats, planes ? f_hi : nullptr, planes ? f_lo : nullptr, T,
                          sums, dev, st, rows);
    }
    if (rc) return rc;
    rc = model_forward(packed, D, L, planes ? nullptr : feats, f_hi, f_lo, B, T, prob, w, ws_bytes - used, st);
    if (rc) return rc;
    if (bin) return binarize_launch(prob, nullptr, T, B, *bin, row_base, dec, counts, seg_off, seg, cap, st);
    rc = threshold_median_launch(prob, B, T, thr, kernel, dec, 1, nullptr, 0.f, st);
    if (rc) return rc;
    return segments_launch(dec, nullptr, T, B, sinc ? 1 : 2, row_base, counts, seg_off, seg, cap, st);
}

int b200vad_pipeline_fbank_f32(const void* packed, int L, const float* wav, const int32_t* lens, int B, int64_t N,
                               int64_t stride, float thr, int kernel, float* prob, uint8_t* dec, int32_t* counts,
                               int64_t* seg_off, int32_t* seg, int64_t cap, void* ws, size_t ws_bytes, void* stream) {
    B200VAD_CHECK_ARG(B >= 0 && B <= 65535 && N >= 1 && stride >= 1, "bad shape");
    return pipeline_run(packed, nullptr, L, wav, 0, lens, B, N, stride, thr, kernel, nullptr, 0, prob, dec, counts, seg_off, seg, cap, ws,
                        ws_bytes, (cudaStream_t)stream);
}

int b200vad_pipeline_fbank_i16(const void* packed, int L, const int16_t* wav, const int32_t* lens, int B, int64_t N,
                               int64_t stride, float thr, int kernel, float* prob, uint8_t* dec, int32_t* counts,
                               int64_t* seg_off, int32_t* seg, int64_t cap, void* ws, size_t ws_bytes, void* stream) {
    B200VAD_CHECK_ARG(B >= 0 && B <= 65535 && N >= 1 && stride >= 1, "bad shape");
    return pipeline_run(packed, nullptr, L, wav, 1, lens, B, N, stride, thr, kernel, nullptr, 0, prob, dec, counts, seg_off, seg, cap, ws,
                        ws_bytes, (cudaStream_t)stream);
}

static int pipeline_sincnet_entry(const void* packed, const void* sinc, int L, const void* wav, int wav_i16, int B, int64_t N,
                                  int64_t stride, float thr, int kernel, float* prob, uint8_t* dec, int32_t* counts, int64_t* seg_off,
                                  int32_t* seg, int64_t cap, void* ws, size_t ws_bytes, void* stream) {
    B200VAD_CHECK_ARG(sinc, "null pointer");
    B200VAD_CHECK_ARG(L > 0 && B >= 0 && B <= 65535 && stride >= 1 && cap >= 0, "bad shape");
    B200VAD_CHECK_ARG(N >= 991, "waveform shorter than the SincNet receptive field (991 samples)");
    return pipeline_run(packed, sinc, L, wav, wav_i16, nullptr, B, N, stride, thr, kernel, nullptr, 0, prob, dec, counts, seg_off, seg, cap, ws,
                        ws_bytes, (cudaStream_t)stream);
}
int b200vad_pipeline_sincnet_f32(const void* packed_model, const void* packed_sincnet, int num_layers, const float* wav, int B,
                                 int64_t N, int64_t wav_stride, float thr, int kernel, float* prob, uint8_t* dec, int32_t* counts,
                                 int64_t* seg_off, int32_t* seg, int64_t cap, void* ws, size_t ws_bytes, void* stream) {
    return pipeline_sincnet_entry(packed_model, packed_sincnet, num_layers, wav, 0, B, N, wav_stride, thr, kernel, prob, dec, counts,
                                  seg_off, seg, cap, ws, ws_bytes, stream);
}
int b200vad_pipeline_sincnet_i16(const void* packed_model, const void* packed_sincnet, int num_layers, const int16_t* wav, int B,
                                 int64_t N, int64_t wav_stride, float thr, int kernel, float* prob, uint8_t* dec, int32_t* counts,
                                 int64_t* seg_off, int32_t* seg, int64_t cap, void* ws, size_t ws_bytes, void* stream) {
    return pipeline_sincnet_entry(packed_model, packed_sincnet, num_layers, wav, 1, B, N, wav_stride, thr, kernel, prob, dec, counts,
                                  seg_off, seg, cap, ws, ws_bytes, stream);
}

int b200vad_pipeline_binarize(const void* packed_model, const void* packed_sincnet, int num_layers, const void* wav, int wav_i16,
                              const int32_t* lens, int B, int64_t N, int64_t wav_stride, const b200vad_binarize_params* params,
                              float* prob, uint8_t* dec, int32_t* counts, int64_t* seg_off, int32_t* seg, int64_t cap, void* ws,
                              size_t ws_bytes, void* stream) {
    int rc = check_binarize(params);
    if (rc) return rc;
    B200VAD_CHECK_ARG(num_layers > 0 && B >= 0 && B <= 65535 && N >= 1 && wav_stride >= 1 && cap >= 0, "bad shape");
    if (packed_sincnet) {
        B200VAD_CHECK_ARG(!lens, "the SincNet path takes no lens");
        B200VAD_CHECK_ARG(N >= 991, "waveform shorter than the SincNet receptive field (991 samples)");
    }
    return pipeline_run(packed_model, packed_sincnet, num_layers, wav, wav_i16 != 0, lens, B, N, wav_stride, 0.f, 0, params, 0, prob,
                        dec, counts, seg_off, seg, cap, ws, ws_bytes, (cudaStream_t)stream);
}

int b200vad_pipeline_rows(const void* packed_model, const void* packed_sincnet, int num_layers, const void* const* rows, int wav_i16,
                          const int32_t* lens, int B, int64_t N, float thr, int kernel, const b200vad_binarize_params* params,
                          float* prob, uint8_t* dec, int32_t* counts, int64_t* seg_off, int32_t* seg, int64_t cap, void* ws,
                          size_t ws_bytes, void* stream) {
    if (params) {
        int rc = check_binarize(params);
        if (rc) return rc;
    }
    B200VAD_CHECK_ARG(num_layers > 0 && B >= 0 && B <= 65535 && N >= 1 && cap >= 0, "bad shape");
    B200VAD_CHECK_ARG(!packed_sincnet || N >= 991, "waveform shorter than the SincNet receptive field (991 samples)");
    if (B == 0) return B200VAD_OK;
    B200VAD_CHECK_ARG(rows && lens, "null pointer");
    return pipeline_run(packed_model, packed_sincnet, num_layers, nullptr, wav_i16 != 0, lens, B, N, 1, thr, kernel, params, 0, prob, dec,
                        counts, seg_off, seg, cap, ws, ws_bytes, (cudaStream_t)stream, rows);
}

// ---------------------------------------------------------------- host-buffer session
// Two slots, three streams (H2D / compute / D2H).  submit() only enqueues; wait() blocks on the slot's D2H
// event.  With a batch in flight in each slot the H2D copy of batch i+1 and the D2H of batch i-1 overlap
// the compute of batch i.
struct SessionSlot {
    float* wav_dev;
    float* prob_dev;
    uint8_t* dec_dev;
    int32_t* counts_dev;
    int64_t* seg_off_dev;
    int32_t* seg_dev;
    int64_t* total_host;    // pinned
    cudaEvent_t copy_begin, copied, compute_begin, computed, drained;
    int B;                  // rows in flight (0 = free)
};
struct b200vad_session {
    int device;
    const void* packed;
    const void* sinc;       // packed SincNet blob (SincNet -> PyanNet path), or null (fbank -> PyanNet2)
    int L;
    int chunk;
    int64_t N, T, max_seg_per_row;
    bool bin_on;            // b200vad_session_set_binarize
    b200vad_binarize_params bin;
    cudaStream_t copy_stream, compute_stream, d2h_stream, seg_stream;
    cudaEvent_t epoch;      // recorded at creation; slot event times are reported relative to it
    SessionSlot slot[2];
    void* ws;
    size_t ws_bytes;
};

static int session_create(int device, const void* packed_device, const void* sinc, int num_layers, int max_chunk_rows, int64_t N,
                          b200vad_session** out) {
    B200VAD_CHECK_ARG(out && packed_device, "null pointer");
    B200VAD_CHECK_ARG(num_layers > 0 && max_chunk_rows > 0 && max_chunk_rows <= 65535 && N >= 1, "bad shape");
    B200VAD_CHECK_ARG(!sinc || N >= 991, "waveform shorter than the SincNet receptive field (991 samples)");
    int rc = b200vad_init(device);
    if (rc) return rc;
    b200vad_session* s = new b200vad_session();
    memset(s, 0, sizeof(*s));
    s->device = device; s->packed = packed_device; s->sinc = sinc; s->L = num_layers; s->chunk = max_chunk_rows; s->N = N;
    s->T = fe_frames(sinc != nullptr, N);
    // segments per row at most: ceil(T / 2) single-frame runs (the SincNet RLE, binarization); the fbank RLE needs ceil(T / 3)
    s->max_seg_per_row = (s->T + 1) / 2;
    cudaError_t e = cudaSuccess;
    auto ok = [&](cudaError_t r) { if (e == cudaSuccess) e = r; };
    ok(cudaStreamCreateWithFlags(&s->copy_stream, cudaStreamNonBlocking));
    ok(cudaStreamCreateWithFlags(&s->compute_stream, cudaStreamNonBlocking));
    ok(cudaStreamCreateWithFlags(&s->d2h_stream, cudaStreamNonBlocking));
    ok(cudaStreamCreateWithFlags(&s->seg_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
        SessionSlot& sl = s->slot[i];
        ok(cudaEventCreate(&sl.copy_begin));
        ok(cudaEventCreate(&sl.copied));
        ok(cudaEventCreate(&sl.compute_begin));
        ok(cudaEventCreate(&sl.computed));
        ok(cudaEventCreate(&sl.drained));
        ok(cudaMalloc(&sl.wav_dev, sizeof(float) * (size_t)s->chunk * N));
        ok(cudaMalloc(&sl.prob_dev, sizeof(float) * (size_t)s->chunk * s->T));
        ok(cudaMalloc(&sl.dec_dev, (size_t)s->chunk * s->T));
        ok(cudaMalloc(&sl.counts_dev, sizeof(int32_t) * s->chunk));
        ok(cudaMalloc(&sl.seg_off_dev, sizeof(int64_t) * (s->chunk + 1)));
        ok(cudaMalloc(&sl.seg_dev, sizeof(int32_t) * 3 * (size_t)s->chunk * s->max_seg_per_row));
        ok(cudaMallocHost(&sl.total_host, sizeof(int64_t)));
    }
    s->ws_bytes = pipeline_ws_bytes(s->chunk, N, sinc != nullptr);
    ok(cudaMalloc(&s->ws, s->ws_bytes));
    ok(cudaEventCreate(&s->epoch));
    ok(cudaEventRecord(s->epoch, s->copy_stream));
    if (e != cudaSuccess) {
        set_error("b200vad_session_create: %s", cudaGetErrorString(e));
        b200vad_session_destroy(s);
        return e == cudaErrorMemoryAllocation ? B200VAD_ENOMEM : B200VAD_ECUDA;
    }
    *out = s;
    return B200VAD_OK;
}
int b200vad_session_create(int device, const void* packed_device, int num_layers, int max_chunk_rows, int64_t N,
                           b200vad_session** out) {
    return session_create(device, packed_device, nullptr, num_layers, max_chunk_rows, N, out);
}
int b200vad_session_create_sincnet(int device, const void* packed_model, const void* packed_sincnet, int num_layers,
                                   int max_chunk_rows, int64_t N, b200vad_session** out) {
    B200VAD_CHECK_ARG(packed_sincnet, "null pointer");
    return session_create(device, packed_model, packed_sincnet, num_layers, max_chunk_rows, N, out);
}

static int session_submit(b200vad_session* s, int slot, const void* wav_host, int wav_i16, int B, int row_base, float thr, int kernel,
                          uint8_t* dec_host, float* prob_host) {
    SessionSlot& sl = s->slot[slot];
    const int64_t N = s->N, T = s->T;
    B200VAD_CUDA(cudaEventRecord(sl.copy_begin, s->copy_stream));
    B200VAD_CUDA(cudaMemcpyAsync(sl.wav_dev, wav_host, (wav_i16 ? sizeof(int16_t) : sizeof(float)) * (size_t)B * N,
                                 cudaMemcpyHostToDevice, s->copy_stream));
    B200VAD_CUDA(cudaEventRecord(sl.copied, s->copy_stream));
    B200VAD_CUDA(cudaStreamWaitEvent(s->compute_stream, sl.copied, 0));
    B200VAD_CUDA(cudaEventRecord(sl.compute_begin, s->compute_stream));
    int rc = pipeline_run(s->packed, s->sinc, s->L, sl.wav_dev, wav_i16, nullptr, B, N, N, thr, kernel, s->bin_on ? &s->bin : nullptr,
                          row_base, sl.prob_dev, sl.dec_dev,
                          sl.counts_dev, sl.seg_off_dev, sl.seg_dev, (int64_t)B * s->max_seg_per_row, s->ws, s->ws_bytes,
                          s->compute_stream);
    if (rc) return rc;
    B200VAD_CUDA(cudaEventRecord(sl.computed, s->compute_stream));
    B200VAD_CUDA(cudaStreamWaitEvent(s->d2h_stream, sl.computed, 0));
    B200VAD_CUDA(cudaMemcpyAsync(sl.total_host, sl.seg_off_dev + B, sizeof(int64_t), cudaMemcpyDeviceToHost, s->d2h_stream));
    if (dec_host)
        B200VAD_CUDA(cudaMemcpyAsync(dec_host, sl.dec_dev, (size_t)B * T, cudaMemcpyDeviceToHost, s->d2h_stream));
    if (prob_host)
        B200VAD_CUDA(cudaMemcpyAsync(prob_host, sl.prob_dev, sizeof(float) * (size_t)B * T, cudaMemcpyDeviceToHost, s->d2h_stream));
    B200VAD_CUDA(cudaEventRecord(sl.drained, s->d2h_stream));
    sl.B = B;
    return B200VAD_OK;
}

// blocks until the slot's results are on the host; copies at most `cap` segment triples, *nseg = segments found
static int session_wait(b200vad_session* s, int slot, int32_t* seg_host, int64_t cap, int64_t* nseg) {
    SessionSlot& sl = s->slot[slot];
    B200VAD_CUDA(cudaEventSynchronize(sl.drained));
    const int64_t n = *sl.total_host;
    const int64_t take = std::max<int64_t>(0, std::min<int64_t>(n, cap));
    if (take > 0) {
        // own stream: d2h_stream may already hold the other slot's copies, which wait for that slot's compute
        B200VAD_CUDA(cudaMemcpyAsync(seg_host, sl.seg_dev, sizeof(int32_t) * 3 * take, cudaMemcpyDeviceToHost, s->seg_stream));
        B200VAD_CUDA(cudaStreamSynchronize(s->seg_stream));
    }
    sl.B = 0;
    *nseg = n;
    return B200VAD_OK;
}

static int submit_entry(b200vad_session* s, int slot, const void* wav_host, int wav_i16, int B, float thr, int kernel,
                        uint8_t* dec_host, float* prob_host) {
    B200VAD_CHECK_ARG(s && wav_host, "null pointer");
    B200VAD_CHECK_ARG(slot == 0 || slot == 1, "slot must be 0 or 1");
    B200VAD_CHECK_ARG(B >= 1 && B <= s->chunk, "B must be in [1, max_chunk_rows]");
    if (s->slot[slot].B != 0) {
        set_error("session_submit_host: slot %d still holds an unwaited batch", slot);
        return B200VAD_ESTATE;
    }
    B200VAD_CUDA(cudaSetDevice(s->device));
    return session_submit(s, slot, wav_host, wav_i16, B, 0, thr, kernel, dec_host, prob_host);
}
int b200vad_session_submit_host(b200vad_session* s, int slot, const float* wav_host, int B, float thr, int kernel,
                                uint8_t* dec_host, float* prob_host) {
    return submit_entry(s, slot, wav_host, 0, B, thr, kernel, dec_host, prob_host);
}
int b200vad_session_submit_host_i16(b200vad_session* s, int slot, const int16_t* wav_host, int B, float thr, int kernel,
                                    uint8_t* dec_host, float* prob_host) {
    return submit_entry(s, slot, wav_host, 1, B, thr, kernel, dec_host, prob_host);
}

int b200vad_session_wait(b200vad_session* s, int slot, int32_t* seg_host, int64_t cap, int64_t* nseg) {
    B200VAD_CHECK_ARG(s && nseg && (seg_host || cap == 0), "null pointer");
    B200VAD_CHECK_ARG((slot == 0 || slot == 1) && cap >= 0, "bad slot / cap");
    if (s->slot[slot].B == 0) {
        set_error("session_wait: slot %d has no batch in flight", slot);
        return B200VAD_ESTATE;
    }
    B200VAD_CUDA(cudaSetDevice(s->device));
    return session_wait(s, slot, seg_host, cap, nseg);
}

int b200vad_session_set_binarize(b200vad_session* s, const b200vad_binarize_params* params) {
    B200VAD_CHECK_ARG(s, "null pointer");
    if (params) {
        int rc = check_binarize(params);
        if (rc) return rc;
        s->bin = *params;
    }
    s->bin_on = params != nullptr;
    return B200VAD_OK;
}

int b200vad_session_slot_times(b200vad_session* s, int slot, float* ms) {
    B200VAD_CHECK_ARG(s && ms && (slot == 0 || slot == 1), "bad argument");
    SessionSlot& sl = s->slot[slot];
    cudaEvent_t ev[5] = {sl.copy_begin, sl.copied, sl.compute_begin, sl.computed, sl.drained};
    B200VAD_CUDA(cudaEventSynchronize(sl.drained));
    for (int i = 0; i < 5; ++i) B200VAD_CUDA(cudaEventElapsedTime(ms + i, s->epoch, ev[i]));
    return B200VAD_OK;
}

int b200vad_session_run_host(b200vad_session* s, const float* wav_host, int B, float thr, int kernel, uint8_t* dec_host,
                             float* prob_host, int32_t* seg_host, int64_t cap, int64_t* nseg) {
    B200VAD_CHECK_ARG(s && wav_host && nseg && (seg_host || cap == 0), "null pointer");
    B200VAD_CHECK_ARG(B >= 0 && cap >= 0, "bad size");
    *nseg = 0;
    if (B == 0) return B200VAD_OK;
    if (s->slot[0].B != 0 || s->slot[1].B != 0) {
        set_error("session_run_host: a submitted batch is still in flight");
        return B200VAD_ESTATE;
    }
    B200VAD_CUDA(cudaSetDevice(s->device));
    const int nchunks = (B + s->chunk - 1) / s->chunk;
    const int64_t N = s->N, T = s->T;
    int64_t total = 0;
    auto drain = [&](int c) -> int {
        int64_t n = 0;
        int rc = session_wait(s, c & 1, seg_host ? seg_host + 3 * std::min(total, cap) : nullptr,
                              std::max<int64_t>(0, cap - total), &n);
        total += n;
        return rc;
    };
    for (int c = 0; c < nchunks; ++c) {
        const int b0 = c * s->chunk, bc = std::min(s->chunk, B - b0);
        int rc;
        if (c >= 2 && (rc = drain(c - 2))) return rc;
        rc = session_submit(s, c & 1, wav_host + (size_t)b0 * N, 0, bc, b0, thr, kernel,
                            dec_host ? dec_host + (size_t)b0 * T : nullptr, prob_host ? prob_host + (size_t)b0 * T : nullptr);
        if (rc) return rc;
    }
    for (int c = std::max(0, nchunks - 2); c < nchunks; ++c) {
        int rc = drain(c);
        if (rc) return rc;
    }
    *nseg = total;
    return B200VAD_OK;
}

void b200vad_session_destroy(b200vad_session* s) {
    if (!s) return;
    cudaSetDevice(s->device);
    if (s->compute_stream) cudaStreamSynchronize(s->compute_stream);
    if (s->d2h_stream) cudaStreamSynchronize(s->d2h_stream);
    for (int i = 0; i < 2; ++i) {
        SessionSlot& sl = s->slot[i];
        if (sl.wav_dev) cudaFree(sl.wav_dev);
        if (sl.prob_dev) cudaFree(sl.prob_dev);
        if (sl.dec_dev) cudaFree(sl.dec_dev);
        if (sl.counts_dev) cudaFree(sl.counts_dev);
        if (sl.seg_off_dev) cudaFree(sl.seg_off_dev);
        if (sl.seg_dev) cudaFree(sl.seg_dev);
        if (sl.total_host) cudaFreeHost(sl.total_host);
        if (sl.copy_begin) cudaEventDestroy(sl.copy_begin);
        if (sl.compute_begin) cudaEventDestroy(sl.compute_begin);
        if (sl.copied) cudaEventDestroy(sl.copied);
        if (sl.computed) cudaEventDestroy(sl.computed);
        if (sl.drained) cudaEventDestroy(sl.drained);
    }
    if (s->ws) cudaFree(s->ws);
    if (s->epoch) cudaEventDestroy(s->epoch);
    if (s->copy_stream) cudaStreamDestroy(s->copy_stream);
    if (s->compute_stream) cudaStreamDestroy(s->compute_stream);
    if (s->d2h_stream) cudaStreamDestroy(s->d2h_stream);
    if (s->seg_stream) cudaStreamDestroy(s->seg_stream);
    delete s;
}

// ---------------------------------------------------------------- streaming session (BASELINE config 5)
// Every stream keeps its last `window` samples in a double-write ring; push() appends `hop` new samples per
// stream and runs the whole path on the buffered windows, so the newest frames equal the batch path applied to
// the same window (the BiLSTM is non-causal: there is no cheaper exact update, SURVEY 8a "streaming").
// The per-push kernel sequence is fixed, so it is captured once into a CUDA graph and replayed.
struct b200vad_stream {
    int device;
    const void* packed;
    const void* sinc;       // packed SincNet blob, or null (fbank front end)
    int L, S, hop, nf, pos;
    int64_t W, T;
    float thr;
    int kernel;
    bool bin_on;            // b200vad_stream_set_binarize
    b200vad_binarize_params bin;
    bool use_graph;
    cudaStream_t st;
    cudaGraph_t graph;
    cudaGraphExec_t exec;
    cudaEvent_t e0, e1;
    float *ring, *lin, *chunk, *feats, *prob, *prob_new, *prob_new_host;
    double* sums;
    uint8_t *dec, *dec_new, *dec_new_host;
    int32_t *counts, *seg;  // binarization: per-stream region counts and triples (S * ceil(T / 2))
    int64_t* seg_off;
    void* ws;
    size_t ws_bytes;
    // speech events (b200vad_stream_set_events): device state (S, 5) and flush mask (S); one buffer holding ev (S, nf + 1, 2)
    // then ev_counts (S), copied to its pinned twin by one copy per push; the drained triples queue on the host
    bool ev_on;
    b200vad_binarize_params evp;
    int64_t* ev_state;
    uint8_t *ev_flush, *ev_flush_host;
    void *ev_dev, *ev_host;
    int64_t pushes;         // pushes so far; stream i's timeline holds (pushes - born[i]) * nf frames
    int64_t *born, *ev_base; // per stream: push at which its timeline began, timeline frame of its event tracking's frame 0
    int64_t *ev_list, ev_n, ev_cap;
};

static inline size_t stream_ev_bytes(const b200vad_stream* s) { return sizeof(int64_t) * (size_t)s->S * (s->nf + 1) * 2; }

// warm_up: the events step runs on 0 frames, which leaves its state as it is
static int stream_forward(b200vad_stream* s, bool warm_up = false) {
    const int D = fe_dim(s->sinc != nullptr);
    __half* f_hi = reinterpret_cast<__half*>(s->feats);
    __half* f_lo = f_hi + (size_t)s->S * s->T * round8(D);
    int rc = s->sinc ? sincnet_forward(s->sinc, s->lin, 0, s->S, s->W, s->W, nullptr, f_hi, f_lo, s->ws, s->ws_bytes, s->st)
                     : fbank_launch(s->lin, 0, nullptr, s->S, s->W, s->W, nullptr, f_hi, f_lo, s->T, s->sums, s->device, s->st);
    if (rc) return rc;
    rc = model_forward(s->packed, D, s->L, nullptr, f_hi, f_lo, s->S, s->T, s->prob, s->ws, s->ws_bytes, s->st);
    if (rc) return rc;
    rc = s->bin_on ? binarize_launch(s->prob, nullptr, s->T, s->S, s->bin, 0, s->dec, s->counts, s->seg_off, s->seg,
                                     (int64_t)s->S * ((s->T + 1) / 2), s->st)
                   : threshold_median_launch(s->prob, s->S, s->T, s->thr, s->kernel, s->dec, 1, nullptr, 0.f, s->st);
    if (rc) return rc;
    rc = stream_newest_launch(s->prob, s->dec, s->S, s->T, s->nf, s->prob_new, s->dec_new, s->st);
    if (rc || !s->ev_on) return rc;
    int64_t* ev = static_cast<int64_t*>(s->ev_dev);
    return regions_step_launch(s->prob_new, s->S, warm_up ? 0 : s->nf, s->nf, s->evp, s->ev_state, nullptr, ev,
                               reinterpret_cast<int32_t*>(reinterpret_cast<char*>(ev) + stream_ev_bytes(s)), s->nf + 1, s->st);
}

// after the events of one call are in ev_host: queue them as (stream, kind, timeline frame) triples, in stream then frame order
static int stream_queue_events(b200vad_stream* s) {
    const int64_t* ev = static_cast<const int64_t*>(s->ev_host);
    const int32_t* counts = reinterpret_cast<const int32_t*>(static_cast<const char*>(s->ev_host) + stream_ev_bytes(s));
    for (int i = 0; i < s->S; ++i) {
        for (int j = 0; j < counts[i]; ++j) {
            if (s->ev_n == s->ev_cap) {
                const int64_t cap = std::max<int64_t>(1024, 2 * s->ev_cap);
                int64_t* p = static_cast<int64_t*>(realloc(s->ev_list, sizeof(int64_t) * 3 * cap));
                if (!p) { set_error("stream events: out of host memory"); return B200VAD_ENOMEM; }
                s->ev_list = p; s->ev_cap = cap;
            }
            const int64_t* e = ev + ((int64_t)i * (s->nf + 1) + j) * 2;
            int64_t* o = s->ev_list + 3 * s->ev_n++;
            o[0] = i; o[1] = e[1]; o[2] = s->ev_base[i] + e[0];
        }
    }
    return B200VAD_OK;
}

// end the groups of the streams in ev_flush_host under the current policy (events on), and queue their end events.  Blocking.
static int stream_flush_events(b200vad_stream* s) {
    B200VAD_CUDA(cudaMemcpyAsync(s->ev_flush, s->ev_flush_host, s->S, cudaMemcpyHostToDevice, s->st));
    int64_t* ev = static_cast<int64_t*>(s->ev_dev);
    int rc = regions_step_launch(nullptr, s->S, 0, 0, s->evp, s->ev_state, s->ev_flush, ev,
                                 reinterpret_cast<int32_t*>(reinterpret_cast<char*>(ev) + stream_ev_bytes(s)), s->nf + 1, s->st);
    if (rc) return rc;
    B200VAD_CUDA(cudaMemcpyAsync(s->ev_host, s->ev_dev, stream_ev_bytes(s) + sizeof(int32_t) * s->S, cudaMemcpyDeviceToHost, s->st));
    B200VAD_CUDA(cudaStreamSynchronize(s->st));
    return stream_queue_events(s);
}

static int stream_capture(b200vad_stream* s) {
    if (s->exec) { cudaGraphExecDestroy(s->exec); s->exec = nullptr; }
    if (s->graph) { cudaGraphDestroy(s->graph); s->graph = nullptr; }
    int rc = stream_forward(s, true);                   // warm-up: one-time function attributes, table init
    if (rc) return rc;
    B200VAD_CUDA(cudaStreamSynchronize(s->st));
    B200VAD_CUDA(cudaStreamBeginCapture(s->st, cudaStreamCaptureModeThreadLocal));
    rc = stream_forward(s);
    cudaError_t e = cudaStreamEndCapture(s->st, &s->graph);
    if (rc) return rc;
    if (e != cudaSuccess) { set_error("stream capture failed: %s", cudaGetErrorString(e)); return B200VAD_ECUDA; }
    B200VAD_CUDA(cudaGraphInstantiate(&s->exec, s->graph, 0));
    return B200VAD_OK;
}

static int stream_create(int device, const void* packed_device, const void* sinc, int num_layers, int num_streams,
                         int64_t window_samples, int hop_samples, int use_graph, b200vad_stream** out) {
    B200VAD_CHECK_ARG(out && packed_device, "null pointer");
    B200VAD_CHECK_ARG(num_layers > 0 && num_streams > 0 && num_streams <= 65535, "bad shape");
    if (sinc) {
        // frames of consecutive windows fall on one grid only when the hop is a whole number of SincNet frame steps
        B200VAD_CHECK_ARG(hop_samples > 0 && hop_samples % kSincStep == 0 && window_samples >= 991 && window_samples >= hop_samples &&
                              window_samples <= (1 << 30) && hop_samples / kSincStep <= sinc_dims(window_samples).P3,
                          "SincNet streaming: hop must be a multiple of 270 samples, window >= 991 samples, hop <= window");
    } else {
        B200VAD_CHECK_ARG(hop_samples > 0 && hop_samples % kFrameShift == 0 && window_samples % kFrameShift == 0 &&
                              window_samples >= hop_samples && window_samples <= (1 << 30),
                          "window and hop must be multiples of 160 samples, hop <= window");
    }
    int rc = b200vad_init(device);
    if (rc) return rc;
    b200vad_stream* s = new b200vad_stream();
    memset(s, 0, sizeof(*s));
    s->device = device; s->packed = packed_device; s->sinc = sinc; s->L = num_layers; s->S = num_streams; s->hop = hop_samples;
    s->W = window_samples; s->T = fe_frames(sinc != nullptr, window_samples); s->nf = hop_samples / (sinc ? kSincStep : kFrameShift);
    s->thr = 0.5f; s->kernel = 49; s->use_graph = use_graph != 0;
    cudaError_t e = cudaSuccess;
    auto ok = [&](cudaError_t r) { if (e == cudaSuccess) e = r; };
    const size_t S = s->S, W = s->W, T = s->T;
    ok(cudaStreamCreateWithFlags(&s->st, cudaStreamNonBlocking));
    ok(cudaEventCreate(&s->e0)); ok(cudaEventCreate(&s->e1));
    ok(cudaMalloc(&s->ring, sizeof(float) * S * 2 * W));
    ok(cudaMalloc(&s->lin, sizeof(float) * S * W));
    ok(cudaMalloc(&s->chunk, sizeof(float) * S * s->hop));
    ok(cudaMalloc(&s->feats, sizeof(float) * S * T * round8(fe_dim(sinc != nullptr))));
    ok(cudaMalloc(&s->sums, sizeof(double) * S));
    ok(cudaMalloc(&s->prob, sizeof(float) * S * T));
    ok(cudaMalloc(&s->dec, S * T));
    ok(cudaMalloc(&s->prob_new, sizeof(float) * S * s->nf));
    ok(cudaMalloc(&s->dec_new, S * s->nf));
    ok(cudaMalloc(&s->counts, sizeof(int32_t) * S));
    ok(cudaMalloc(&s->seg_off, sizeof(int64_t) * (S + 1)));
    ok(cudaMalloc(&s->seg, sizeof(int32_t) * 3 * S * ((T + 1) / 2)));
    ok(cudaMallocHost(&s->prob_new_host, sizeof(float) * S * s->nf));
    ok(cudaMallocHost(&s->dec_new_host, S * s->nf));
    ok(cudaMalloc(&s->ev_state, sizeof(int64_t) * S * 5));
    ok(cudaMalloc(&s->ev_flush, S));
    ok(cudaMallocHost(&s->ev_flush_host, S));
    ok(cudaMalloc(&s->ev_dev, stream_ev_bytes(s) + sizeof(int32_t) * S));
    ok(cudaMallocHost(&s->ev_host, stream_ev_bytes(s) + sizeof(int32_t) * S));
    s->born = static_cast<int64_t*>(calloc(S, sizeof(int64_t)));
    s->ev_base = static_cast<int64_t*>(calloc(S, sizeof(int64_t)));
    if (!s->born || !s->ev_base) ok(cudaErrorMemoryAllocation);
    s->ws_bytes = b200vad_model_workspace_bytes(s->S, s->T);
    if (sinc)   // the front end's workspace is dead before the model runs on the same stream
        s->ws_bytes = std::max(s->ws_bytes, (size_t)std::min<int64_t>(s->S, sinc_chunk_rows(s->W)) * sinc_ws_per_row(s->W) + 4096);
    ok(cudaMalloc(&s->ws, s->ws_bytes));
    if (e == cudaSuccess) ok(cudaMemsetAsync(s->ring, 0, sizeof(float) * S * 2 * W, s->st));
    if (e == cudaSuccess) ok(cudaMemsetAsync(s->lin, 0, sizeof(float) * S * W, s->st));
    if (e == cudaSuccess) ok(cudaMemsetAsync(s->ev_state, 0, sizeof(int64_t) * S * 5, s->st));
    if (e != cudaSuccess) {
        set_error("b200vad_stream_create: %s", cudaGetErrorString(e));
        b200vad_stream_destroy(s);
        return e == cudaErrorMemoryAllocation ? B200VAD_ENOMEM : B200VAD_ECUDA;
    }
    if (s->use_graph && (rc = stream_capture(s))) { b200vad_stream_destroy(s); return rc; }
    *out = s;
    return B200VAD_OK;
}
int b200vad_stream_create(int device, const void* packed_device, int num_layers, int num_streams, int64_t window_samples,
                          int hop_samples, int use_graph, b200vad_stream** out) {
    return stream_create(device, packed_device, nullptr, num_layers, num_streams, window_samples, hop_samples, use_graph, out);
}
int b200vad_stream_create_sincnet(int device, const void* packed_model, const void* packed_sincnet, int num_layers, int num_streams,
                                  int64_t window_samples, int hop_samples, int use_graph, b200vad_stream** out) {
    B200VAD_CHECK_ARG(packed_sincnet, "null pointer");
    return stream_create(device, packed_model, packed_sincnet, num_layers, num_streams, window_samples, hop_samples, use_graph, out);
}

int b200vad_stream_push(b200vad_stream* s, const float* chunk, int chunk_on_host, float thr, int kernel, float* prob_new_host,
                        uint8_t* dec_new_host, float* device_ms) {
    B200VAD_CHECK_ARG(s && chunk, "null pointer");
    B200VAD_CHECK_ARG(s->bin_on || (kernel >= 1 && (kernel & 1)), "median kernel must be odd");
    B200VAD_CUDA(cudaSetDevice(s->device));
    int rc;
    if (!s->bin_on && (thr != s->thr || kernel != s->kernel)) {
        s->thr = thr; s->kernel = kernel;
        if (s->use_graph && (rc = stream_capture(s))) return rc;
    }
    B200VAD_CUDA(cudaEventRecord(s->e0, s->st));
    const float* src = chunk;
    if (chunk_on_host) {
        B200VAD_CUDA(cudaMemcpyAsync(s->chunk, chunk, sizeof(float) * (size_t)s->S * s->hop, cudaMemcpyHostToDevice, s->st));
        src = s->chunk;
    }
    if ((rc = stream_append_launch(s->ring, src, s->lin, s->S, (int)s->W, s->hop, s->pos, s->st))) return rc;
    s->pos += s->hop;
    if (s->pos >= s->W) s->pos -= (int)s->W;
    if (s->use_graph) {
        B200VAD_CUDA(cudaGraphLaunch(s->exec, s->st));
    } else if ((rc = stream_forward(s))) {
        return rc;
    }
    const size_t n = (size_t)s->S * s->nf;
    B200VAD_CUDA(cudaMemcpyAsync(s->prob_new_host, s->prob_new, sizeof(float) * n, cudaMemcpyDeviceToHost, s->st));
    B200VAD_CUDA(cudaMemcpyAsync(s->dec_new_host, s->dec_new, n, cudaMemcpyDeviceToHost, s->st));
    if (s->ev_on)
        B200VAD_CUDA(cudaMemcpyAsync(s->ev_host, s->ev_dev, stream_ev_bytes(s) + sizeof(int32_t) * s->S, cudaMemcpyDeviceToHost, s->st));
    B200VAD_CUDA(cudaEventRecord(s->e1, s->st));
    B200VAD_CUDA(cudaEventSynchronize(s->e1));
    ++s->pushes;
    if (prob_new_host) memcpy(prob_new_host, s->prob_new_host, sizeof(float) * n);
    if (dec_new_host) memcpy(dec_new_host, s->dec_new_host, n);
    if (s->ev_on && (rc = stream_queue_events(s))) return rc;
    if (device_ms) B200VAD_CUDA(cudaEventElapsedTime(device_ms, s->e0, s->e1));
    return B200VAD_OK;
}

int b200vad_stream_set_binarize(b200vad_stream* s, const b200vad_binarize_params* params) {
    B200VAD_CHECK_ARG(s, "null pointer");
    if (params) {
        int rc = check_binarize(params);
        if (rc) return rc;
        s->bin = *params;
    }
    s->bin_on = params != nullptr;
    B200VAD_CUDA(cudaSetDevice(s->device));
    return s->use_graph ? stream_capture(s) : B200VAD_OK;
}

int b200vad_stream_set_events(b200vad_stream* s, const b200vad_binarize_params* params) {
    B200VAD_CHECK_ARG(s, "null pointer");
    if (params) {
        int rc = check_binarize(params);
        if (rc) return rc;
    }
    B200VAD_CUDA(cudaSetDevice(s->device));
    if (s->ev_on) {             // end every stream's open group under the old policy; this zeroes the state
        memset(s->ev_flush_host, 1, s->S);
        int rc = stream_flush_events(s);
        if (rc) return rc;
    }
    s->ev_on = params != nullptr;
    if (params) s->evp = *params;
    for (int i = 0; i < s->S; ++i) s->ev_base[i] = (s->pushes - s->born[i]) * s->nf;
    return s->use_graph ? stream_capture(s) : B200VAD_OK;
}

int b200vad_stream_end(b200vad_stream* s, const int32_t* streams, int n) {
    B200VAD_CHECK_ARG(s && (streams || n == 0), "null pointer");
    B200VAD_CHECK_ARG(n >= 0 && n <= s->S, "bad count");
    memset(s->ev_flush_host, 0, s->S);
    for (int j = 0; j < n; ++j) {
        B200VAD_CHECK_ARG(streams[j] >= 0 && streams[j] < s->S, "stream index out of range");
        B200VAD_CHECK_ARG(!s->ev_flush_host[streams[j]], "repeated stream index");
        s->ev_flush_host[streams[j]] = 1;
    }
    if (n == 0) return B200VAD_OK;
    B200VAD_CUDA(cudaSetDevice(s->device));
    if (s->ev_on) {
        int rc = stream_flush_events(s);
        if (rc) return rc;
    }
    for (int j = 0; j < n; ++j) {
        const int i = streams[j];
        B200VAD_CUDA(cudaMemsetAsync(s->ring + (size_t)i * 2 * s->W, 0, sizeof(float) * 2 * s->W, s->st));
        B200VAD_CUDA(cudaMemsetAsync(s->lin + (size_t)i * s->W, 0, sizeof(float) * s->W, s->st));
        s->born[i] = s->pushes;
        s->ev_base[i] = 0;
    }
    B200VAD_CUDA(cudaStreamSynchronize(s->st));
    return B200VAD_OK;
}

int b200vad_stream_events(b200vad_stream* s, int64_t* ev_host, int64_t cap, int64_t* n) {
    B200VAD_CHECK_ARG(s && n && (ev_host || cap == 0) && cap >= 0, "bad argument");
    if (!ev_host) { *n = s->ev_n; return B200VAD_OK; }
    const int64_t k = std::min(cap, s->ev_n);
    if (k == 0) { *n = 0; return B200VAD_OK; }
    memcpy(ev_host, s->ev_list, sizeof(int64_t) * 3 * k);
    memmove(s->ev_list, s->ev_list + 3 * k, sizeof(int64_t) * 3 * (s->ev_n - k));
    s->ev_n -= k;
    *n = k;
    return B200VAD_OK;
}

/* debugging / parity: copy the current buffered windows (S, window) and all frame outputs to the host */
int b200vad_stream_snapshot(b200vad_stream* s, float* window_host, float* prob_host, uint8_t* dec_host) {
    B200VAD_CHECK_ARG(s, "null pointer");
    B200VAD_CUDA(cudaSetDevice(s->device));
    B200VAD_CUDA(cudaStreamSynchronize(s->st));
    if (window_host) B200VAD_CUDA(cudaMemcpy(window_host, s->lin, sizeof(float) * (size_t)s->S * s->W, cudaMemcpyDeviceToHost));
    if (prob_host) B200VAD_CUDA(cudaMemcpy(prob_host, s->prob, sizeof(float) * (size_t)s->S * s->T, cudaMemcpyDeviceToHost));
    if (dec_host) B200VAD_CUDA(cudaMemcpy(dec_host, s->dec, (size_t)s->S * s->T, cudaMemcpyDeviceToHost));
    return B200VAD_OK;
}

void b200vad_stream_destroy(b200vad_stream* s) {
    if (!s) return;
    cudaSetDevice(s->device);
    if (s->st) cudaStreamSynchronize(s->st);
    if (s->exec) cudaGraphExecDestroy(s->exec);
    if (s->graph) cudaGraphDestroy(s->graph);
    void* dev_ptrs[] = {s->ring, s->lin, s->chunk, s->feats, s->sums, s->prob, s->dec, s->prob_new, s->dec_new, s->counts, s->seg_off,
                        s->seg, s->ws, s->ev_state, s->ev_flush, s->ev_dev};
    for (void* p : dev_ptrs) if (p) cudaFree(p);
    void* host_ptrs[] = {s->prob_new_host, s->dec_new_host, s->ev_flush_host, s->ev_host};
    for (void* p : host_ptrs) if (p) cudaFreeHost(p);
    free(s->born); free(s->ev_base); free(s->ev_list);
    if (s->e0) cudaEventDestroy(s->e0);
    if (s->e1) cudaEventDestroy(s->e1);
    if (s->st) cudaStreamDestroy(s->st);
    delete s;
}

}  // extern "C"
