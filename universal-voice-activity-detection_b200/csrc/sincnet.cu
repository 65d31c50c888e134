// SincNet front-end pieces (src/models/blocks/sincnet.py:34-103), channel-last layout.
//
//   wav (B,N) --InstanceNorm1d(1)--> (B,N) --sinc conv 80x251 /10, abs--> (B,L1,80)
//   --MaxPool3 + InstanceNorm(80) + leaky_relu--> (B,P1,80) --Conv1d(80,60,5)--> (B,L2,60)
//   --pool/norm/lrelu--> (B,P2,60) --Conv1d(60,60,5)--> (B,L3,60) --pool/norm/lrelu--> (B,Ts,60)
//
// Activations are kept time-major / channel-fastest so that (a) every convolution is the
// overlapping-row GEMM of gemm.cu, and (b) the final (B,Ts,60) tensor already is the LSTM
// input of PyanNet.forward (PyanNet.py:178 rearrange "b f t -> b t f") with no transpose.
// InstanceNorm statistics (biased variance over time per (batch, channel), eps 1e-5) are
// accumulated in double while the max-pool output is written, then applied in place together
// with the affine transform and LeakyReLU(0.01).
#include "kernels.cuh"
#include <algorithm>

namespace b200vad {

// ---------------------------------------------------------------- sinc filter synthesis
// asteroid-filterbanks 0.4 ParamSincFB.filters(): 40 cos + 40 sin band-pass filters of 251 taps.
// low_hz_, band_hz_: (40); window_: (125); n_: (125).  out: (80, 251) fp32.
__global__ void sinc_filters_kernel(const float* __restrict__ low_hz_, const float* __restrict__ band_hz_,
                                    const float* __restrict__ window_, const float* __restrict__ n_, float* __restrict__ out) {
    const int f = blockIdx.x;          // 0..39
    const int j = threadIdx.x;         // 0..125 (125 = centre tap)
    const float min_low = 50.f, min_band = 50.f, nyq = 8000.f;
    float low = min_low + fabsf(low_hz_[f]);
    float high = fminf(fmaxf(low + min_band + fabsf(band_hz_[f]), min_low), nyq);
    float band = high - low;
    float inv = 2.f * band;
    float* cosf_row = out + (size_t)f * 251;
    float* sinf_row = out + (size_t)(40 + f) * 251;
    if (j == 125) {
        cosf_row[125] = (2.f * band) / inv;
        sinf_row[125] = 0.f / inv;
        return;
    }
    if (j > 125) return;
    float n = n_[j], w = window_[j];
    float ft_low = low * n, ft_high = high * n;
    float cl = ((sinf(ft_high) - sinf(ft_low)) / (n / 2.f)) * w;
    float sl = ((cosf(ft_low) - cosf(ft_high)) / (n / 2.f)) * w;
    cosf_row[j] = cl / inv;
    cosf_row[250 - j] = cl / inv;
    sinf_row[j] = sl / inv;
    sinf_row[250 - j] = (-sl) / inv;
}
int sinc_filters_launch(const float* low, const float* band, const float* window, const float* n, float* out, cudaStream_t s) {
    sinc_filters_kernel<<<40, 128, 0, s>>>(low, band, window, n, out);
    B200VAD_LAUNCH_CHECK();
    return B200VAD_OK;
}

// Conv1d weight (Cout, Cin, k) -> GEMM weight (Cout, k*Cin) matching channel-last rows
__global__ void repack_conv_kernel(const float* __restrict__ w, int Cout, int Cin, int k, float* __restrict__ out) {
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    int tot = Cout * Cin * k;
    if (idx >= tot) return;
    int co = idx / (Cin * k), rem = idx % (Cin * k), kk = rem / Cin, ci = rem % Cin;
    out[idx] = w[((size_t)co * Cin + ci) * k + kk];
}
int repack_conv_launch(const float* w, int Cout, int Cin, int k, float* out, cudaStream_t s) {
    int tot = Cout * Cin * k;
    repack_conv_kernel<<<(tot + 255) / 256, 256, 0, s>>>(w, Cout, Cin, k, out);
    B200VAD_LAUNCH_CHECK();
    return B200VAD_OK;
}

// ---------------------------------------------------------------- waveform instance norm
// Samples are fp32, or 16-bit PCM converted as an audio loader does (int16 / 32768, exact): every later operation sees the
// same floats, so the output from int16 input equals the output from the converted fp32 waveform bit for bit.
__device__ __forceinline__ float sample_f32(float v) { return v; }
__device__ __forceinline__ float sample_f32(int16_t v) { return (float)v * (1.f / 32768.f); }

// Rows of N samples, at wav + b * stride or, with a pointer table, at rows[b] (windows of several recordings in one launch).
// With a table, lens[b] are the row's valid samples and every sample at index >= lens[b] is read as 0 without touching
// memory: that is the zero-padded tail window of the reference, which the InstanceNorm sees.  The statistics walk all N
// samples in the same order either way, and adding 0 changes no partial sum, so the statistics and planes of a row read
// through the table equal those of the same samples copied into a zero-padded row, bit for bit.
template <typename S>
__device__ __forceinline__ const S* wave_row(const S* wav, const S* const* rows, int64_t stride, int b) {
    return rows ? rows[b] : wav + (int64_t)b * stride;
}
__device__ __forceinline__ int64_t wave_valid(const int32_t* lens, int64_t N, int b) {
    return lens ? min((int64_t)lens[b], N) : N;
}

// stats[b] = (sum, sumsq) in double
template <typename S>
__global__ void __launch_bounds__(256) wave_stats_kernel(const S* __restrict__ wav, const S* const* __restrict__ rows,
                                                         const int32_t* __restrict__ lens, int64_t N, int64_t stride,
                                                         double* __restrict__ stats) {
    const int b = blockIdx.y;
    const S* row = wave_row(wav, rows, stride, b);
    const int64_t n = wave_valid(lens, N, b);
    const int64_t chunk = 256 * 32;
    int64_t begin = (int64_t)blockIdx.x * chunk, end = min(begin + chunk, N);
    float s = 0.f, q = 0.f;
    for (int64_t i = begin + threadIdx.x; i < end; i += 256) {
        float v = i < n ? sample_f32(__ldg(row + i)) : 0.f;
        s += v;
        q = fmaf(v, v, q);
    }
    double ds = s, dq = q;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        ds += __shfl_xor_sync(0xffffffffu, ds, o);
        dq += __shfl_xor_sync(0xffffffffu, dq, o);
    }
    __shared__ double ps[8], pq[8];
    if ((threadIdx.x & 31) == 0) { ps[threadIdx.x >> 5] = ds; pq[threadIdx.x >> 5] = dq; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0, c = 0;
        for (int i = 0; i < 8; ++i) { a += ps[i]; c += pq[i]; }
        atomicAdd(stats + 2 * b, exact_partial<32>(a));        // exact additions -> independent of the CTA order (common.cuh)
        atomicAdd(stats + 2 * b + 1, exact_partial<32>(c));
    }
}
__global__ void __launch_bounds__(256) wave_norm_kernel(const float* __restrict__ wav, int64_t N, int64_t stride,
                                                        const double* __restrict__ stats, const float* __restrict__ gamma,
                                                        const float* __restrict__ beta, float* __restrict__ out) {
    const int b = blockIdx.y;
    double mean = stats[2 * b] / (double)N;
    double var = stats[2 * b + 1] / (double)N - mean * mean;
    float rstd = (float)(1.0 / sqrt(fmax(var, 0.0) + 1e-5));
    float m = (float)mean, g = gamma[0], be = beta[0];
    const float* row = wav + (int64_t)b * stride;
    float* o = out + (int64_t)b * N;
    for (int64_t i = (int64_t)blockIdx.x * 256 * 16 + threadIdx.x; i < min(N, ((int64_t)blockIdx.x + 1) * 256 * 16); i += 256)
        o[i] = (row[i] - m) * rstd * g + be;
}
int wave_instnorm_launch(const float* wav, int B, int64_t N, int64_t stride, const float* gamma, const float* beta,
                         double* stats, float* out, cudaStream_t s) {
    { int rc = zero_f64_launch(stats, (int64_t)2 * B, s); if (rc) return rc; }
    dim3 g1((unsigned)((N + 8191) / 8192), B);
    wave_stats_kernel<float><<<g1, 256, 0, s>>>(wav, nullptr, nullptr, N, stride, stats);
    B200VAD_LAUNCH_CHECK();
    dim3 g2((unsigned)((N + 4095) / 4096), B);
    wave_norm_kernel<<<g2, 256, 0, s>>>(wav, N, stride, stats, gamma, beta, out);
    B200VAD_LAUNCH_CHECK();
    return B200VAD_OK;
}

// normalised waveform as fp16 (hi, lo) planes in FOUR shifted copies (shift 0, 2, 4, 6 samples), each (B, Np):
// copy e holds wn[i + 2 e].  The sinc convolution has stride 10 samples = 20 bytes, which is not a legal TMA row
// stride; but rows t = 4 m + r of one residue class r start at 40 m + 10 r = (40 m + 8 floor(10 r / 8)) + (10 r mod 8),
// i.e. at a 16-byte aligned offset of the copy shifted by 10 r mod 8 in {0, 2, 4, 6}, 80 bytes apart: four
// overlapping-row tensor maps, one per residue class, feed the tcgen05 GEMM without an im2col pass.
// 8 samples row[i .. i + 7] as floats with 16-byte loads (vec_ok: 16-byte aligned rows)
__device__ __forceinline__ void load8_f32(const float* row, float (&v)[8]) {
    const float4 a0 = __ldg(reinterpret_cast<const float4*>(row)), a1 = __ldg(reinterpret_cast<const float4*>(row + 4));
    v[0] = a0.x; v[1] = a0.y; v[2] = a0.z; v[3] = a0.w; v[4] = a1.x; v[5] = a1.y; v[6] = a1.z; v[7] = a1.w;
}
__device__ __forceinline__ void load8_f32(const int16_t* row, float (&v)[8]) {
    const uint4 a = __ldg(reinterpret_cast<const uint4*>(row));
    const uint32_t w[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        v[2 * j] = sample_f32((int16_t)(w[j] & 0xffffu));
        v[2 * j + 1] = sample_f32((int16_t)(w[j] >> 16));
    }
}
template <typename S>
__global__ void __launch_bounds__(256) wave_norm_planes_kernel(const S* __restrict__ wav, const S* const* __restrict__ rows,
                                                               const int32_t* __restrict__ lens, int64_t N, int64_t stride, int64_t Np,
                                                               int B, const double* __restrict__ stats, const float* __restrict__ gamma,
                                                               const float* __restrict__ beta, __half* __restrict__ hi,
                                                               __half* __restrict__ lo, float s1) {
    const int b = blockIdx.y;
    double mean = stats[2 * b] / (double)N;
    double var = stats[2 * b + 1] / (double)N - mean * mean;
    float rstd = (float)(1.0 / sqrt(fmax(var, 0.0) + 1e-5));
    float m = (float)mean, g = gamma[0], be = beta[0];
    const S* row = wave_row(wav, rows, stride, b);
    const int64_t n = wave_valid(lens, N, b);
    // 8 consecutive samples per thread (Np and the copies' bases are multiples of 8 elements): copy e receives them at
    // element i - 2 e, i.e. at a 16 / 4 / 8 / 4-byte aligned address for e = 0 / 1 / 2 / 3
    const bool vec_ok = rows ? (reinterpret_cast<uintptr_t>(row) & 15) == 0
                             : ((stride * (int64_t)sizeof(S)) % 16 == 0) && ((reinterpret_cast<uintptr_t>(wav) & 15) == 0);
    for (int64_t i = ((int64_t)blockIdx.x * 256 + threadIdx.x) * 8; i < Np + 8; i += (int64_t)gridDim.x * 256 * 8) {
        float v[8];
        if (vec_ok && i + 8 <= n) {
            load8_f32(row + i, v);
        } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = (i + j < n) ? sample_f32(row[i + j]) : 0.f;
        }
        __align__(16) __half h[8], l[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            h[j] = __float2half_rn(0.f); l[j] = h[j];
            if (i + j < N) split_scaled_f16((v[j] - m) * rstd * g + be, s1, h[j], l[j]);
        }
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int64_t d = i - 2 * e;                      // copy e: element d holds sample d + 2 e
            __half* dh = hi + ((int64_t)e * B + b) * Np;
            __half* dl = lo + ((int64_t)e * B + b) * Np;
            if (d >= 0 && d + 8 <= Np) {
                if (e == 0) {
                    *reinterpret_cast<uint4*>(dh + d) = *reinterpret_cast<const uint4*>(h);
                    *reinterpret_cast<uint4*>(dl + d) = *reinterpret_cast<const uint4*>(l);
                } else if (e == 2) {
                    *reinterpret_cast<uint2*>(dh + d) = *reinterpret_cast<const uint2*>(h);
                    *reinterpret_cast<uint2*>(dh + d + 4) = *reinterpret_cast<const uint2*>(h + 4);
                    *reinterpret_cast<uint2*>(dl + d) = *reinterpret_cast<const uint2*>(l);
                    *reinterpret_cast<uint2*>(dl + d + 4) = *reinterpret_cast<const uint2*>(l + 4);
                } else {
#pragma unroll
                    for (int j = 0; j < 8; j += 2) {
                        *reinterpret_cast<uint32_t*>(dh + d + j) = *reinterpret_cast<const uint32_t*>(h + j);
                        *reinterpret_cast<uint32_t*>(dl + d + j) = *reinterpret_cast<const uint32_t*>(l + j);
                    }
                }
            } else {
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    if (d + j >= 0 && d + j < Np) { dh[d + j] = h[j]; dl[d + j] = l[j]; }
            }
        }
    }
}
template <typename S>
static int wave_norm_planes_run(const S* wav, const S* const* rows, const int32_t* lens, int B, int64_t N, int64_t stride, int64_t Np,
                                const float* gamma, const float* beta, double* stats, __half* hi, __half* lo, cudaStream_t s,
                                int scaled_planes) {
    { int rc = zero_f64_launch(stats, (int64_t)2 * B, s); if (rc) return rc; }
    dim3 g1((unsigned)((N + 8191) / 8192), B);
    wave_stats_kernel<S><<<g1, 256, 0, s>>>(wav, rows, lens, N, stride, stats);
    B200VAD_LAUNCH_CHECK();
    dim3 g2((unsigned)((Np + 8 + 2047) / 2048), B);
    wave_norm_planes_kernel<S><<<g2, 256, 0, s>>>(wav, rows, lens, N, stride, Np, B, stats, gamma, beta, hi, lo,
                                                  scaled_planes ? 1.f - kPlaneScale : 1.f);
    B200VAD_LAUNCH_CHECK();
    return B200VAD_OK;
}
int wave_norm_planes_launch(const void* wav, int wav_i16, int B, int64_t N, int64_t stride, int64_t Np, const float* gamma,
                            const float* beta, double* stats, __half* hi, __half* lo, cudaStream_t s, int scaled_planes,
                            const void* const* rows, const int32_t* lens) {
    if (wav_i16)
        return wave_norm_planes_run(reinterpret_cast<const int16_t*>(wav), reinterpret_cast<const int16_t* const*>(rows), lens, B, N, stride,
                                    Np, gamma, beta, stats, hi, lo, s, scaled_planes);
    return wave_norm_planes_run(reinterpret_cast<const float*>(wav), reinterpret_cast<const float* const*>(rows), lens, B, N, stride, Np,
                                gamma, beta, stats, hi, lo, s, scaled_planes);
}

// GEMM weights for the tcgen05 path, zero padded to 128 output rows: (Cout, K) -> (128, ld)
__global__ void pad_rows_kernel(const float* __restrict__ w, int Cout, int K, int ld, float* __restrict__ out) {
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= 128 * ld) return;
    int r = idx / ld, k = idx % ld;
    out[idx] = (r < Cout && k < K) ? w[(size_t)r * K + k] : 0.f;
}
int pad_rows_launch(const float* w, int Cout, int K, int ld, float* out, cudaStream_t s) {
    pad_rows_kernel<<<(128 * ld + 255) / 256, 256, 0, s>>>(w, Cout, K, ld, out);
    B200VAD_LAUNCH_CHECK();
    return B200VAD_OK;
}
// Conv1d weight (Cout, Cin, k) -> (128, ld) with element [co][kk * Cp + ci] (channel-last rows whose channels are padded to Cp)
__global__ void repack_conv_pad_kernel(const float* __restrict__ w, int Cout, int Cin, int k, int Cp, int ld, float* __restrict__ out) {
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= 128 * ld) return;
    int co = idx / ld, col = idx % ld, kk = col / Cp, ci = col % Cp;
    out[idx] = (co < Cout && kk < k && ci < Cin) ? w[((size_t)co * Cin + ci) * k + kk] : 0.f;
}
int repack_conv_pad_launch(const float* w, int Cout, int Cin, int k, int Cp, int ld, float* out, cudaStream_t s) {
    repack_conv_pad_kernel<<<(128 * ld + 255) / 256, 256, 0, s>>>(w, Cout, Cin, k, Cp, ld, out);
    B200VAD_LAUNCH_CHECK();
    return B200VAD_OK;
}

// ---------------------------------------------------------------- MaxPool1d(3,3) + InstanceNorm stats
// in: (B, L, C) -> pooled (B, P, C), P = L / 3 (floor).  stats[(b*C + c)*2 + {0,1}] += sum, sumsq.
constexpr int kPoolRows = 64;   // pooled rows per CTA
__global__ void __launch_bounds__(256) pool_stats_kernel(const float* __restrict__ in, int64_t L, int C, int64_t P,
                                                         float* __restrict__ pooled, double* __restrict__ stats) {
    const int b = blockIdx.y;
    const int lanes = 256 / C;                 // row lanes (3 for C=80, 4 for C=60)
    const int c = threadIdx.x % C, rl = threadIdx.x / C;
    const int64_t p0 = (int64_t)blockIdx.x * kPoolRows;
    float s = 0.f, q = 0.f;
    if (rl < lanes) {
        for (int64_t p = p0 + rl; p < min(P, p0 + kPoolRows); p += lanes) {
            const float* src = in + ((int64_t)b * L + 3 * p) * C + c;
            float v = fmaxf(fmaxf(__ldg(src), __ldg(src + C)), __ldg(src + 2 * C));
            pooled[((int64_t)b * P + p) * C + c] = v;
            s += v;
            q = fmaf(v, v, q);
        }
    }
    __shared__ float ss[256], sq[256];
    ss[threadIdx.x] = s;
    sq[threadIdx.x] = q;
    __syncthreads();
    if (threadIdx.x < C) {
        double a = 0, d = 0;
        for (int r = 0; r < lanes; ++r) { a += ss[r * C + threadIdx.x]; d += sq[r * C + threadIdx.x]; }
        atomicAdd(stats + ((int64_t)b * C + threadIdx.x) * 2, exact_partial<32>(a));
        atomicAdd(stats + ((int64_t)b * C + threadIdx.x) * 2 + 1, exact_partial<32>(d));
    }
}
// x = leaky_relu((x - mean) * rstd * gamma + beta): written in place as fp32, or -- when planes are given -- only as fp16
// (hi, lo) planes (B, P, Cp) with the channels zero padded to Cp (the operand of the next convolution on the tcgen05 path;
// the fp32 copy has no reader there).  Four channels per thread (C % 4 == 0, Cp % 4 == 0).
__global__ void __launch_bounds__(256) norm_lrelu_kernel(float* __restrict__ x, int64_t P, int C, const double* __restrict__ stats,
                                                         const float* __restrict__ gamma, const float* __restrict__ beta,
                                                         __half* __restrict__ p_hi, __half* __restrict__ p_lo, int Cp, float s1) {
    const int b = blockIdx.y;
    __shared__ float sc[128], sh[128];
    if (threadIdx.x < C) {
        double mean = stats[((int64_t)b * C + threadIdx.x) * 2] / (double)P;
        double var = stats[((int64_t)b * C + threadIdx.x) * 2 + 1] / (double)P - mean * mean;
        float rstd = (float)(1.0 / sqrt(fmax(var, 0.0) + 1e-5));
        float g = gamma[threadIdx.x];
        sc[threadIdx.x] = rstd * g;
        sh[threadIdx.x] = beta[threadIdx.x] - (float)mean * rstd * g;
    }
    __syncthreads();
    const int q = (p_hi ? Cp : C) / 4;                        // 4-channel groups per row (including the padding groups)
    const int64_t groups = P * q;
    float* base = x + (int64_t)b * P * C;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < groups; i += (int64_t)gridDim.x * 256) {
        const int64_t r = i / q;
        const int c = (int)(i - r * q) * 4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (c < C) {
            v = *reinterpret_cast<const float4*>(base + r * C + c);
            v.x = fmaf(v.x, sc[c], sh[c]); v.y = fmaf(v.y, sc[c + 1], sh[c + 1]);
            v.z = fmaf(v.z, sc[c + 2], sh[c + 2]); v.w = fmaf(v.w, sc[c + 3], sh[c + 3]);
            v.x = v.x > 0.f ? v.x : 0.01f * v.x; v.y = v.y > 0.f ? v.y : 0.01f * v.y;
            v.z = v.z > 0.f ? v.z : 0.01f * v.z; v.w = v.w > 0.f ? v.w : 0.01f * v.w;
        }
        if (p_hi) {
            __align__(8) __half h[4], l[4];
            split_scaled_f16(v.x, s1, h[0], l[0]); split_scaled_f16(v.y, s1, h[1], l[1]);
            split_scaled_f16(v.z, s1, h[2], l[2]); split_scaled_f16(v.w, s1, h[3], l[3]);
            const int64_t o = ((int64_t)b * P + r) * Cp + c;
            *reinterpret_cast<uint2*>(p_hi + o) = *reinterpret_cast<const uint2*>(h);
            *reinterpret_cast<uint2*>(p_lo + o) = *reinterpret_cast<const uint2*>(l);
        } else {
            *reinterpret_cast<float4*>(base + r * C + c) = v;
        }
    }
}
int norm_lrelu_launch(float* pooled, int B, int64_t P, int C, const double* stats, const float* gamma, const float* beta,
                      cudaStream_t s, __half* p_hi, __half* p_lo, int Cp, int scaled_planes) {
    if (P <= 0 || B == 0) return B200VAD_OK;
    if (C > 128 || C < 1 || C % 4 != 0 || (p_hi && (Cp % 4 != 0 || Cp < C))) {
        set_error("norm_lrelu: C in [1,128], C and Cp multiples of 4, Cp >= C");
        return B200VAD_EINVAL;
    }
    const int64_t groups = P * ((p_hi ? Cp : C) / 4);
    dim3 g2((unsigned)std::min<int64_t>((groups + 1023) / 1024, 65535), B);
    norm_lrelu_kernel<<<g2, 256, 0, s>>>(pooled, P, C, stats, gamma, beta, p_hi, p_lo, Cp, scaled_planes ? 1.f - kPlaneScale : 1.f);
    B200VAD_LAUNCH_CHECK();
    return B200VAD_OK;
}

int pool_norm_lrelu_launch(const float* in, int B, int64_t L, int C, float* pooled, double* stats, const float* gamma,
                           const float* beta, cudaStream_t s, __half* p_hi, __half* p_lo, int Cp, int scaled_planes) {
    if (C > 128 || C < 1) {
        set_error("pool_norm: C must be in [1,128]");
        return B200VAD_EINVAL;
    }
    const int64_t P = L / 3;
    if (P <= 0 || B == 0) return B200VAD_OK;
    { int rc = zero_f64_launch(stats, (int64_t)2 * B * C, s); if (rc) return rc; }
    dim3 g1((unsigned)((P + kPoolRows - 1) / kPoolRows), B);
    pool_stats_kernel<<<g1, 256, 0, s>>>(in, L, C, P, pooled, stats);
    B200VAD_LAUNCH_CHECK();
    return norm_lrelu_launch(pooled, B, P, C, stats, gamma, beta, s, p_hi, p_lo, Cp, scaled_planes);
}

}  // namespace b200vad
