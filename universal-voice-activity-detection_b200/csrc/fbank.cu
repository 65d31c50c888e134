// Fused lhotse-style log-mel filterbank for sm_100a.
//
// Replaces the ~10 ATen kernels + cuFFT + SGEMM of lhotse Wav2LogFilterBank that the
// reference calls at src/utils/helper.py:120-130 and src/datasets/*/utils.py
// (e.g. ami/utils.py:152-163): whole-signal DC removal, whole-signal pre-emphasis 0.97,
// mirror padding (snip_edges=False), 400/160 framing, povey window, zero-pad to 512,
// real FFT, power spectrum, 80 Kaldi mel triangles, log(max(., eps)).
//
// One CTA (128 threads) = 32 consecutive frames of one utterance.  The pre-emphasised span
// (31*160+400 samples) is staged once in shared memory with float4 loads, so every
// waveform sample is read from HBM once (plus the 5 % tile halo, an L2 hit).
// FFT: 512-point real FFT as a 256-point complex FFT, 16 threads per frame, two
// radix-16 passes held in registers with one padded shared-memory transpose between
// them; real-FFT untangling on conjugate pairs (k, 256-k) + |X|^2, the sparse mel
// triangles and the log, all inside the frame's own half-warp (no CTA barriers).
// HBM traffic per frame: 640 B in + 320 B out = 960 B (algorithmic); intermediates
// (frames, spectrum, power) never leave the SM.  The kernel is FP32-issue bound, not HBM
// bound: ~13 k thread-instructions per frame (DESIGN.md section 4).
#include "kernels.cuh"
#include <math.h>
#include <stdio.h>
#include <mutex>

namespace b200vad {

constexpr int kTileFrames = 32;
constexpr int kSpan = (kTileFrames - 1) * kFrameShift + kFrameLen;   // 5360 samples
constexpr int kFbankThreads = 128;
constexpr int kGroups = kFbankThreads / 16;                           // 16 threads per frame
constexpr int kZStride = 17 * 16;                                     // padded 16x16 complex tile (float2 units)
constexpr int kPowStride = 264;
constexpr int kMaxMelWidth = 32;
static const int kSlotTapsHost[kNumMel / 16] = {3, 4, 6, 10, 16};      // widest triangle per slot of 16 mel bins
constexpr int kMelRows = 18;                                          // widest Kaldi triangle at 512/16 kHz spans 17 FFT bins

struct FbankTables {
    float window[kFrameLen];
    float2 tw256[256];          // exp(-2*pi*i*m/256)
    float2 tw512[257];          // exp(-2*pi*i*k/512), k = 0..256
    float2 tw16[16][16];        // stage twiddles W256^(j*k1) as [k1][j] (coalesced per half-warp)
    int mel_start[kNumMel];
    int mel_len[kNumMel];
    float mel_w[kNumMel][kMaxMelWidth];
    float mel_wt[kMelRows][kNumMel];      // transposed: [k_rel][bin], zero beyond a bin's width
};

static FbankTables* g_tables_dev[64] = {nullptr};
static std::mutex g_tables_mu;

static double mel_scale(double f) { return 1127.0 * log(1.0 + f / 700.0); }

// Host-side table construction (double precision, rounded once to fp32).
static void build_tables(FbankTables& t) {
    const double pi = 3.14159265358979323846;
    for (int n = 0; n < kFrameLen; ++n) {
        double hann = 0.5 - 0.5 * cos(2.0 * pi * n / (kFrameLen - 1));
        t.window[n] = (float)pow(hann, 0.85);
    }
    for (int m = 0; m < 256; ++m) t.tw256[m] = make_float2((float)cos(2 * pi * m / 256), (float)-sin(2 * pi * m / 256));
    for (int k1 = 0; k1 < 16; ++k1)
        for (int jj = 0; jj < 16; ++jj)
            t.tw16[k1][jj] = make_float2((float)cos(2 * pi * (jj * k1) / 256), (float)-sin(2 * pi * (jj * k1) / 256));
    for (int k = 0; k <= 256; ++k) t.tw512[k] = make_float2((float)cos(2 * pi * k / 512), (float)-sin(2 * pi * k / 512));
    // Kaldi mel triangles (torchaudio.compliance.kaldi.get_mel_banks, vtln off):
    // 80 bins, 20 Hz .. 7600 Hz, triangles in the mel domain, FFT bin width 31.25 Hz.
    const double lo = mel_scale(20.0), hi = mel_scale(8000.0 - 400.0);
    const double delta = (hi - lo) / (kNumMel + 1);
    for (int b = 0; b < kNumMel; ++b) {
        double left = lo + b * delta, center = lo + (b + 1) * delta, right = lo + (b + 2) * delta;
        int start = -1, len = 0;
        for (int k = 0; k < 256; ++k) {
            double mel = mel_scale(31.25 * k);
            double up = (mel - left) / (center - left), down = (right - mel) / (right - center);
            double w = fmin(up, down);
            if (w > 0.0) {
                if (start < 0) start = k;
                if (k - start < kMaxMelWidth) {
                    t.mel_w[b][k - start] = (float)w;
                    len = k - start + 1;
                }
            }
        }
        t.mel_start[b] = start < 0 ? 0 : start;
        t.mel_len[b] = len;
        for (int j = len; j < kMaxMelWidth; ++j) t.mel_w[b][j] = 0.f;
        for (int j = 0; j < kMelRows; ++j) t.mel_wt[j][b] = (j < len) ? t.mel_w[b][j] : 0.f;
        if (len > kSlotTapsHost[b / 16]) fprintf(stderr, "b200vad: mel triangle %d has %d taps, slot allows %d\n", b, len, kSlotTapsHost[b / 16]);
        if (len > kMelRows) fprintf(stderr, "b200vad: mel triangle %d wider than kMelRows (%d)\n", b, len);
    }
}

int fbank_tables_init(int device) {
    std::lock_guard<std::mutex> lk(g_tables_mu);
    if (device < 0 || device >= 64) return B200VAD_EINVAL;
    if (g_tables_dev[device]) return B200VAD_OK;
    FbankTables* h = new FbankTables();
    build_tables(*h);
    FbankTables* d = nullptr;
    cudaError_t e = cudaMalloc(&d, sizeof(FbankTables));
    if (e == cudaSuccess) e = cudaMemcpy(d, h, sizeof(FbankTables), cudaMemcpyHostToDevice);
    delete h;
    if (e != cudaSuccess) {
        set_error("fbank_tables_init: %s", cudaGetErrorString(e));
        return B200VAD_ECUDA;
    }
    g_tables_dev[device] = d;
    return B200VAD_OK;
}

const FbankTables* fbank_tables(int device) {
    return (device >= 0 && device < 64) ? g_tables_dev[device] : nullptr;
}

// ---------------------------------------------------------------- zero fill
// A kernel instead of cudaMemsetAsync: a memset may be executed by a copy engine, where it queues behind an
// in-flight multi-GB H2D copy of the host session and stalls the whole compute stream (measured: 35 ms per step).
__global__ void zero_f64_kernel(double* __restrict__ p, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = 0.0;
}
int zero_f64_launch(double* p, int64_t n, cudaStream_t stream) {
    if (n <= 0) return B200VAD_OK;
    zero_f64_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(p, n);
    B200VAD_LAUNCH_CHECK();
    return B200VAD_OK;
}

// ---------------------------------------------------------------- waveform loads: fp32 samples or 16-bit PCM
// PCM input is converted exactly as an audio loader does (int16 / 32768 -> float32), so both forms give identical
// features; 16-bit input halves the waveform bytes read (and the H2D copy of the host session).
__device__ __forceinline__ float ld1(const float* p, int64_t i) { return __ldg(p + i); }
__device__ __forceinline__ float ld1(const int16_t* p, int64_t i) { return (float)__ldg(p + i) * (1.f / 32768.f); }
__device__ __forceinline__ float4 ld4(const float* p, int64_t i) { return __ldg(reinterpret_cast<const float4*>(p + i)); }
__device__ __forceinline__ float4 ld4(const int16_t* p, int64_t i) {
    const uint2 u = __ldg(reinterpret_cast<const uint2*>(p + i));
    const short2 a = *reinterpret_cast<const short2*>(&u.x), b = *reinterpret_cast<const short2*>(&u.y);
    const float k = 1.f / 32768.f;
    return make_float4(a.x * k, a.y * k, b.x * k, b.y * k);
}
template <typename WT> __device__ __forceinline__ bool vec_aligned(const WT* p) {
    return (reinterpret_cast<uintptr_t>(p) & (4 * sizeof(WT) - 1)) == 0;
}

// Row b starts at rows[b] when a pointer table is given (windows of several recordings in one launch), else at
// wav + b * stride.  Either way it reads only samples [0, min(lens[b], N)).
template <typename WT>
__device__ __forceinline__ const WT* row_ptr(const WT* wav, const WT* const* rows, int64_t stride, int b) {
    return rows ? rows[b] : wav + (int64_t)b * stride;
}

// ---------------------------------------------------------------- row sums (DC offset)
// grid (chunks, B): fp32 lane partials over <= 32 elements, then double.
template <typename WT>
__global__ void __launch_bounds__(256) row_sum_kernel(const WT* __restrict__ wav, const WT* const* __restrict__ rows,
                                                      const int32_t* __restrict__ lens, int64_t N, int64_t stride,
                                                      double* __restrict__ sums) {
    const int b = blockIdx.y;
    const int64_t n = lens ? min((int64_t)lens[b], N) : N;
    const WT* row = row_ptr(wav, rows, stride, b);
    const int64_t chunk = 256 * 32;
    int64_t begin = (int64_t)blockIdx.x * chunk;
    if (begin >= n) return;
    int64_t end = min(begin + chunk, n);
    double acc = 0.0;
    if (vec_aligned(row) && end - begin == chunk) {
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float4 v = ld4(row, begin + 4 * (threadIdx.x + i * 256));
            s += (v.x + v.y) + (v.z + v.w);
        }
        acc = (double)s;
    } else {
        float s = 0.f;
        for (int64_t i = begin + threadIdx.x; i < end; i += 256) s += ld1(row, i);
        acc = (double)s;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    __shared__ double part[8];
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double tot = 0.0;
#pragma unroll
        for (int i = 0; i < 8; ++i) tot += part[i];
        atomicAdd(sums + b, exact_partial<32>(tot));      // exact additions: the row mean does not depend on the CTA order (common.cuh)
    }
}

// ---------------------------------------------------------------- 16-point FFT in registers
__device__ __forceinline__ float2 cmul(float2 a, float2 b) {
    return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}
__device__ __forceinline__ void fft4(float2& a, float2& b, float2& c, float2& d) {
    // forward DFT-4: outputs in natural order (a,b,c,d) <- (X0,X1,X2,X3)
    float2 s0 = make_float2(a.x + c.x, a.y + c.y), d0 = make_float2(a.x - c.x, a.y - c.y);
    float2 s1 = make_float2(b.x + d.x, b.y + d.y), d1 = make_float2(b.x - d.x, b.y - d.y);
    a = make_float2(s0.x + s1.x, s0.y + s1.y);
    c = make_float2(s0.x - s1.x, s0.y - s1.y);
    // -i * d1 = (d1.y, -d1.x)
    b = make_float2(d0.x + d1.y, d0.y - d1.x);
    d = make_float2(d0.x - d1.y, d0.y + d1.x);
}
// v[n], n = 4a + b  ->  V[k], k = c + 4d (stored back in v[k])
__device__ __forceinline__ void fft16(float2 (&v)[16]) {
    constexpr float C1 = 0.92387953251128674f, S1 = 0.38268343236508977f, C2 = 0.70710678118654752f;
    // W16^m = (cos(2 pi m/16), -sin(2 pi m/16))
    const float2 W[10] = {{1.f, 0.f}, {C1, -S1}, {C2, -C2}, {S1, -C1}, {0.f, -1.f},
                          {-S1, -C1}, {-C2, -C2}, {-C1, -S1}, {-1.f, 0.f}, {-C1, S1}};
#pragma unroll
    for (int b = 0; b < 4; ++b) fft4(v[b], v[4 + b], v[8 + b], v[12 + b]);   // over a; result index c at v[4c+b]
#pragma unroll
    for (int b = 1; b < 4; ++b)
#pragma unroll
        for (int c = 1; c < 4; ++c) v[4 * c + b] = cmul(v[4 * c + b], W[b * c]);
#pragma unroll
    for (int c = 0; c < 4; ++c) fft4(v[4 * c + 0], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);  // over b; result d at v[4c+d]
    // now v[4c + d] holds V[c + 4d]; permute to natural order
    float2 t[16];
#pragma unroll
    for (int c = 0; c < 4; ++c)
#pragma unroll
        for (int d = 0; d < 4; ++d) t[c + 4 * d] = v[4 * c + d];
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = t[i];
}

// ---------------------------------------------------------------- fused fbank kernel
// CTA = 128 threads = 8 groups of 16 threads; a group owns one frame at a time and walks frames g, g+8, g+16, g+24 of
// the 32-frame tile.  After the span is staged there is no CTA barrier: every hand-off (FFT transpose, conjugate
// partners, power spectrum -> mel) stays inside the group's half-warp and needs only __syncwarp.
// Registers are the occupancy limit (5 CTAs = 20 warps per SM at <= 102 registers): the per-thread constants (stage
// twiddles W256^(j k1), untangle twiddles W512^(j+16i), window) are re-read through L1 from 2 KB tables laid out so
// that a half-warp reads one contiguous run, the power spectrum aliases the transpose scratch, and the mel triangles
// use fixed per-slot tap counts (no data-dependent branches).
struct FbankSmem {
    float y[kSpan];                                  // pre-emphasised samples of the tile
    float2 z[kGroups * kZStride];                    // per-group FFT transpose / partner scratch; the power spectrum (x4) of
                                                     // the frame in flight aliases its upper half (float2 slots 136..267)
    float mel_wt[kMelRows][kNumMel];
};
constexpr int kPwOff = 136;                          // first float2 slot of the aliased power spectrum (partners use 0..128)
static_assert(kPwOff * 2 + kPowStride <= kZStride * 2, "power spectrum must fit behind the partner slots");
// widest mel triangle per slot of 16 bins (bins 16 i .. 16 i + 15): fixed, branch-free trip counts; narrower triangles
// read zero weights (the table is zero padded).  Checked against the table at init.
__device__ constexpr int kSlotTaps[kNumMel / 16] = {3, 4, 6, 10, 16};

__device__ __forceinline__ float preemph(float x, float xprev, float mean) {
    // (x - mu) - 0.97 * (xprev - mu), with the reference's separate roundings
    float a = __fsub_rn(x, mean), b = __fsub_rn(xprev, mean);
    return __fsub_rn(a, __fmul_rn(0.97f, b));
}

// PLANES = false: feats (B, T, 80) fp32 (the lhotse layout).  PLANES = true: the same values as fp16 (hi, lo) planes
// feats_hi / feats_lo (B, T, 80) -- the operand format of the layer-0 projection GEMM, so the fused pipeline skips the
// fp32 feature round trip and the split kernel.
template <bool PLANES, typename WT>
__global__ void __launch_bounds__(kFbankThreads, 5)
fbank_kernel(const WT* __restrict__ wav, const WT* const* __restrict__ rows, const int32_t* __restrict__ lens, int64_t N, int64_t stride,
             const double* __restrict__ sums, const FbankTables* __restrict__ tab,
             float* __restrict__ feats, __half* __restrict__ feats_hi, __half* __restrict__ feats_lo, int64_t T_out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    FbankSmem& sm = *reinterpret_cast<FbankSmem*>(smem_raw);
    const int tid = threadIdx.x;
    const int b = blockIdx.y;
    const int64_t n = lens ? min((int64_t)lens[b], N) : N;
    const int64_t T = (n + kFrameShift / 2) / kFrameShift;          // valid frames of this row
    const int64_t f0 = (int64_t)blockIdx.x * kTileFrames;
    const int64_t row_off = ((int64_t)b * T_out) * kNumMel;
    auto put = [&](int64_t idx, float v) {
        if (PLANES) {
            __half h, l;
            split_f16(v, h, l);
            feats_hi[row_off + idx] = h;
            feats_lo[row_off + idx] = l;
        } else {
            feats[row_off + idx] = v;
        }
    };

    if (f0 >= T) {   // tile entirely in the padding: lhotse pads features with LOG_EPSILON
        for (int i = tid; i < kTileFrames * kNumMel; i += kFbankThreads) {
            int64_t f = f0 + i / kNumMel;
            if (f < T_out) put(f * kNumMel + (i % kNumMel), kLogEpsilon);
        }
        return;
    }
    const int nframes = (int)min((int64_t)kTileFrames, T - f0);
    const WT* row = row_ptr(wav, rows, stride, b);
    const float mean = (float)(sums[b] / (double)n);
    const int g = tid >> 4;         // group = frame slot
    const int j = tid & 15;         // lane within the group

    // ---- per-thread constants (registers) and per-CTA tables (smem)
    const float2* const tw = &tab->tw16[0][0] + j;   // W256^(j*k1) at tw[16 * k1], through L1
    const float2* const tq = tab->tw512 + j;      // W512^(j + 16 i): read through L1 (2 KB table, hot)
    const float* const win = tab->window + 2 * j; // povey window, likewise
    int mstart[kNumMel / 16];
#pragma unroll
    for (int i = 0; i < kNumMel / 16; ++i) mstart[i] = __ldg(&tab->mel_start[j + 16 * i]);
    for (int i = tid; i < kMelRows * kNumMel; i += kFbankThreads) (&sm.mel_wt[0][0])[i] = (&tab->mel_wt[0][0])[i];
    // zero the padding behind every group's power spectrum once (fixed-length mel taps may read it with zero weights)
    if (tid < kGroups * 8) reinterpret_cast<float*>(sm.z + (tid >> 3) * kZStride + kPwOff)[257 + (tid & 7)] = 0.f;

    // ---- stage the pre-emphasised span
    const int64_t start = f0 * kFrameShift - kPadLeft;               // original index of span[0]
    const int span = (nframes - 1) * kFrameShift + kFrameLen;
    // interior: every sample read, [start - 1, start + span), lies in [0, n); anything else takes the mirrored path
    const bool interior = (start >= 4) && (start + span <= n) && vec_aligned(row);
    if (interior) {
        // start is a multiple of 8 samples -> aligned 4-sample vector loads
#pragma unroll 4
        for (int i = tid; i < span / 4; i += kFbankThreads) {
            float4 v = ld4(row, start + 4 * i);
            float prev = ld1(row, start + 4 * i - 1);
            float4 o;
            o.x = preemph(v.x, prev, mean);
            o.y = preemph(v.y, v.x, mean);
            o.z = preemph(v.z, v.y, mean);
            o.w = preemph(v.w, v.z, mean);
            *reinterpret_cast<float4*>(&sm.y[4 * i]) = o;
        }
    } else {
        for (int s = tid; s < span; s += kFbankThreads) {
            int64_t i = start + s;
            if (i < 0) i = -1 - i;                 // left mirror (edge sample repeated)
            if (i >= n) i = 2 * n - 1 - i;         // right mirror
            i = max((int64_t)0, min(i, n - 1));
            float x = ld1(row, i);
            float xp = ld1(row, i > 0 ? i - 1 : 0);     // replicate-padded predecessor
            sm.y[s] = preemph(x, xp, mean);
        }
    }
    __syncthreads();

    float2* zf = sm.z + g * kZStride;
    float* pw = reinterpret_cast<float*>(zf + kPwOff);
    for (int pass = 0; pass < kTileFrames / kGroups; ++pass) {
        const int f = pass * kGroups + g;
        const bool active = f < nframes;
        float2 v[16];
        // frames beyond nframes (last tile of a row) compute on stale shared memory and are simply not stored
        {
            const float* ys = sm.y + f * kFrameShift;
            // z[16*n1 + j] = (xw[32*n1 + 2j], xw[32*n1 + 2j + 1]); samples >= 400 are zero padding
#pragma unroll
            for (int n1 = 0; n1 < 16; ++n1) {
                const int s = 32 * n1 + 2 * j;
                if (n1 < 12 || (n1 == 12 && j < 8)) {
                    float2 yy = *reinterpret_cast<const float2*>(ys + s);
                    float2 ww = __ldg(reinterpret_cast<const float2*>(win + 32 * n1));
                    v[n1] = make_float2(yy.x * ww.x, yy.y * ww.y);
                } else {
                    v[n1] = make_float2(0.f, 0.f);
                }
            }
            fft16(v);                                                  // over n1 -> k1
            zf[j] = v[0];
#pragma unroll
            for (int k1 = 1; k1 < 16; ++k1) zf[k1 * 17 + j] = cmul(v[k1], __ldg(tw + 16 * k1));
        }
        __syncwarp();
        {
#pragma unroll
            for (int n2 = 0; n2 < 16; ++n2) v[n2] = zf[j * 17 + n2];    // thread j := k1
            fft16(v);                                                  // over n2 -> k2 ; v[k2] = Z[j + 16*k2]
        }
        __syncwarp();
        {
            // conjugate partners: Z[256 - (j + 16 i)] = Z[(16 - j) + 16 (15 - i)] sits in the upper half (k2 >= 8) of
            // thread 16 - j; slot (k2 - 8) * 16 + j, so the partner of (j, i) is slot (8 - i) * 16 - j (slot 128 = Z[0])
#pragma unroll
            for (int k2 = 8; k2 < 16; ++k2) zf[(k2 - 8) * 16 + j] = v[k2];
            if (j == 0) zf[128] = v[0];
        }
        __syncwarp();
        {
            // real-FFT untangle, two bins per pair: 2Xe = a + conj(c), 2 w^k Xo = T,  4|X[k]|^2 = |2Xe + T|^2,
            // 4|X[256-k]|^2 = |2Xe - T|^2   (a = Z[k], c = Z[256-k], k = j + 16 i)
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float2 a = v[i];
                const float2 c = zf[(8 - i) * 16 - j];
                const float sr = a.x + c.x, si = a.y - c.y;
                const float dr = a.x - c.x, di = a.y + c.y;
                const float2 w = __ldg(tq + 16 * i);
                const float tr = w.x * di + w.y * dr;
                const float ti = w.y * di - w.x * dr;
                const float pr = sr + tr, pi = si + ti, qr = sr - tr, qi = si - ti;
                pw[j + 16 * i] = pr * pr + pi * pi;
                pw[256 - j - 16 * i] = qr * qr + qi * qi;
            }
            if (j == 0) pw[128] = 4.f * (v[8].x * v[8].x + v[8].y * v[8].y);   // X[128] = conj(Z[128])
        }
        __syncwarp();
        // ---- mel triangles + log: lane j owns bins j, j+16, ..., j+64 of its group's frame (64-byte output runs)
        const int64_t fr = f0 + f;
        if (active) {
#pragma unroll
            for (int i = 0; i < kNumMel / 16; ++i) {
                const int m = j + 16 * i;
                const float* p = pw + mstart[i];
                float acc = 0.f;
#pragma unroll
                for (int k = 0; k < kSlotTaps[i]; ++k) acc = fmaf(p[k], sm.mel_wt[k][m], acc);
                put(fr * kNumMel + m, __logf(fmaxf(0.25f * acc, kEpsilon)));
            }
        } else if (fr < T_out) {
#pragma unroll
            for (int i = 0; i < kNumMel / 16; ++i) put(fr * kNumMel + j + 16 * i, kLogEpsilon);
        }
        __syncwarp();
    }
}

// exactly one of feats (fp32) / (feats_hi, feats_lo) (fp16 planes) is written; wav is fp32 or (wav_i16) 16-bit PCM
template <typename WT>
static int fbank_launch_t(const WT* wav, const WT* const* rows, const int32_t* lens, int B, int64_t N, int64_t stride, float* feats,
                          __half* feats_hi, __half* feats_lo, int64_t T_out, double* row_sums, const FbankTables* tab,
                          cudaStream_t stream) {
    int rc;
    if ((rc = set_max_dynamic_smem(reinterpret_cast<const void*>(fbank_kernel<false, WT>), (int)sizeof(FbankSmem)))) return rc;
    if ((rc = set_max_dynamic_smem(reinterpret_cast<const void*>(fbank_kernel<true, WT>), (int)sizeof(FbankSmem)))) return rc;
    if ((rc = zero_f64_launch(row_sums, B, stream))) return rc;
    dim3 g1((unsigned)((N + 256 * 32 - 1) / (256 * 32)), B);
    row_sum_kernel<WT><<<g1, 256, 0, stream>>>(wav, rows, lens, N, stride, row_sums);
    B200VAD_LAUNCH_CHECK();
    dim3 g2((unsigned)((T_out + kTileFrames - 1) / kTileFrames), B);
    prof_begin(3, stream);
    if (feats_hi) fbank_kernel<true, WT><<<g2, kFbankThreads, sizeof(FbankSmem), stream>>>(wav, rows, lens, N, stride, row_sums, tab, nullptr, feats_hi, feats_lo, T_out);
    else fbank_kernel<false, WT><<<g2, kFbankThreads, sizeof(FbankSmem), stream>>>(wav, rows, lens, N, stride, row_sums, tab, feats, nullptr, nullptr, T_out);
    prof_end(3, stream);
    B200VAD_LAUNCH_CHECK();
    return B200VAD_OK;
}

int fbank_launch(const void* wav, int wav_i16, const int32_t* lens, int B, int64_t N, int64_t stride, float* feats, __half* feats_hi,
                 __half* feats_lo, int64_t T_out, double* row_sums, int device, cudaStream_t stream, const void* const* rows) {
    const FbankTables* tab = fbank_tables(device);
    if (!tab) {
        set_error("fbank: b200vad_init(%d) has not been called", device);
        return B200VAD_ESTATE;
    }
    if (B == 0 || T_out == 0) return B200VAD_OK;
    if (wav_i16)
        return fbank_launch_t(static_cast<const int16_t*>(wav), reinterpret_cast<const int16_t* const*>(rows), lens, B, N, stride, feats,
                              feats_hi, feats_lo, T_out, row_sums, tab, stream);
    return fbank_launch_t(static_cast<const float*>(wav), reinterpret_cast<const float* const*>(rows), lens, B, N, stride, feats, feats_hi,
                          feats_lo, T_out, row_sums, tab, stream);
}

}  // namespace b200vad
