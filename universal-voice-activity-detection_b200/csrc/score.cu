// Scoring, long-form stitching and streaming helpers: the integer / byte kernels either side of the model.
//
//  * stat_scores_kernel: tp / fp / tn / fn of the median-filtered decisions against the frame labels
//    (VadModel.test_step, src/engines/vad_engine.py:167-202, torchmetrics BinaryStatScores).
//  * raster_intervals_kernel + count_fa_md_kernel: get_binary_tensor / get_false_alarm /
//    get_missed_detection of src/scripts/predict.py:654-673 on bit masks (32 frames per word): intervals
//    [start_frame, end_frame) are rasterised with atomicOr, false alarms = popc(pred & ~gt), misses = popc(gt & ~pred).
//  * stitch_center_kernel: long-form mode with overlapping windows (BASELINE config 3): the stitched stream takes
//    every frame from the window whose centre is nearest (first / last window keep their outer edge).
//  * stream_append_kernel / stream_newest_kernel: streaming mode (BASELINE config 5): double-write ring buffer of the
//    last `window` samples of every stream, linearised into the staging rows the path runs on.
// All HBM-bound; each byte is read / written once.
#include "kernels.cuh"
#include <algorithm>

namespace b200vad {

// ---------------------------------------------------------------- stat scores
__global__ void __launch_bounds__(256)
stat_scores_kernel(const uint8_t* __restrict__ dec, const uint8_t* __restrict__ lab, int64_t n, unsigned long long* __restrict__ out4) {
    unsigned tp = 0, fp = 0, fn = 0;
    const int64_t nvec = n / 16;
    const bool aligned = (((uintptr_t)dec | (uintptr_t)lab) & 15) == 0;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (aligned) {
        const uint4* d4 = reinterpret_cast<const uint4*>(dec);
        const uint4* l4 = reinterpret_cast<const uint4*>(lab);
        for (int64_t v = i; v < nvec; v += stride) {
            const uint4 d = __ldg(d4 + v), l = __ldg(l4 + v);
            const unsigned dw[4] = {d.x, d.y, d.z, d.w}, lw[4] = {l.x, l.y, l.z, l.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const unsigned dm = __vcmpne4(dw[k], 0u), lm = __vcmpne4(lw[k], 0u);    // 0xff per non-zero byte
                tp += __popc(dm & lm); fp += __popc(dm & ~lm); fn += __popc(~dm & lm);
            }
        }
        tp >>= 3; fp >>= 3; fn >>= 3;
        for (int64_t k = nvec * 16 + i; k < n; k += stride) {
            const bool d = dec[k] != 0, l = lab[k] != 0;
            tp += d && l; fp += d && !l; fn += !d && l;
        }
    } else {
        for (int64_t k = i; k < n; k += stride) {
            const bool d = dec[k] != 0, l = lab[k] != 0;
            tp += d && l; fp += d && !l; fn += !d && l;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        tp += __shfl_xor_sync(0xffffffffu, tp, o);
        fp += __shfl_xor_sync(0xffffffffu, fp, o);
        fn += __shfl_xor_sync(0xffffffffu, fn, o);
    }
    if ((threadIdx.x & 31) == 0) {
        if (tp) atomicAdd(out4 + 0, (unsigned long long)tp);
        if (fp) atomicAdd(out4 + 1, (unsigned long long)fp);
        if (fn) atomicAdd(out4 + 3, (unsigned long long)fn);
    }
}
// tn = n - tp - fp - fn, written by one thread after the counting kernel
__global__ void stat_scores_finish_kernel(unsigned long long* out4, int64_t n) {
    out4[2] = (unsigned long long)n - out4[0] - out4[1] - out4[3];
}
__global__ void zero_u64_kernel(unsigned long long* p, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = 0ull;
}
__global__ void zero_u32_kernel(uint32_t* p, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = 0u;
}

int stat_scores_launch(const uint8_t* dec, const uint8_t* lab, int64_t n, int64_t* out4, cudaStream_t st) {
    unsigned long long* o = reinterpret_cast<unsigned long long*>(out4);
    zero_u64_kernel<<<1, 32, 0, st>>>(o, 4);
    B200VAD_LAUNCH_CHECK();
    if (n > 0) {
        int blocks = (int)std::min<int64_t>((n / 16 + 255) / 256 + 1, 148 * 8);
        stat_scores_kernel<<<blocks, 256, 0, st>>>(dec, lab, n, o);
        B200VAD_LAUNCH_CHECK();
    }
    stat_scores_finish_kernel<<<1, 1, 0, st>>>(o, n);
    B200VAD_LAUNCH_CHECK();
    return B200VAD_OK;
}

// ---------------------------------------------------------------- DER: interval rasterisation + popcounts
// iv: (n, 3) int32 (recording, start_frame, end_frame_exclusive); one warp per interval.
__global__ void __launch_bounds__(256)
raster_intervals_kernel(const int32_t* __restrict__ iv, int64_t n, const int64_t* __restrict__ word_off,
                        const int32_t* __restrict__ nframes, int R, uint32_t* __restrict__ mask) {
    const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= n) return;
    const int r = iv[3 * w];
    if (r < 0 || r >= R) return;
    const int nf = nframes[r];
    // tensor[start:end] = 1 with Python slice clamping (predict.py:660)
    int s = iv[3 * w + 1], e = iv[3 * w + 2];
    if (s < 0) s = max(s + nf, 0);
    if (e < 0) e = max(e + nf, 0);
    s = min(s, nf); e = min(e, nf);
    if (s >= e) return;
    const int w0 = s >> 5, w1 = (e - 1) >> 5;
    uint32_t* base = mask + word_off[r];
    for (int k = w0 + lane; k <= w1; k += 32) {
        uint32_t bits = 0xffffffffu;
        if (k == w0) bits &= 0xffffffffu << (s & 31);
        if (k == w1) bits &= 0xffffffffu >> (31 - ((e - 1) & 31));
        atomicOr(base + k, bits);
    }
}
// grid (chunks, R)
__global__ void __launch_bounds__(256)
count_fa_md_kernel(const uint32_t* __restrict__ gt, const uint32_t* __restrict__ pred, const int64_t* __restrict__ word_off,
                   unsigned long long* __restrict__ fa, unsigned long long* __restrict__ md) {
    const int r = blockIdx.y;
    const int64_t lo = word_off[r], hi = word_off[r + 1];
    unsigned a = 0, m = 0;
    for (int64_t k = lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < hi; k += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t g = __ldg(gt + k), p = __ldg(pred + k);
        a += __popc(p & ~g);
        m += __popc(g & ~p);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        m += __shfl_xor_sync(0xffffffffu, m, o);
    }
    if ((threadIdx.x & 31) == 0) {
        if (a) atomicAdd(fa + r, (unsigned long long)a);
        if (m) atomicAdd(md + r, (unsigned long long)m);
    }
}

int score_intervals_launch(const int32_t* gt_iv, int64_t n_gt, const int32_t* pred_iv, int64_t n_pred, const int64_t* word_off,
                           const int32_t* nframes, int R, int64_t total_words, uint32_t* masks, int64_t* fa, int64_t* md,
                           int max_words_per_rec_hint, cudaStream_t st) {
    if (R <= 0) return B200VAD_OK;
    uint32_t* gmask = masks;
    uint32_t* pmask = masks + total_words;
    if (total_words > 0) {
        zero_u32_kernel<<<(unsigned)((2 * total_words + 255) / 256), 256, 0, st>>>(masks, 2 * total_words);
        B200VAD_LAUNCH_CHECK();
    }
    zero_u64_kernel<<<(unsigned)((R + 255) / 256), 256, 0, st>>>(reinterpret_cast<unsigned long long*>(fa), R);
    B200VAD_LAUNCH_CHECK();
    zero_u64_kernel<<<(unsigned)((R + 255) / 256), 256, 0, st>>>(reinterpret_cast<unsigned long long*>(md), R);
    B200VAD_LAUNCH_CHECK();
    if (n_gt > 0) {
        raster_intervals_kernel<<<(unsigned)((n_gt * 32 + 255) / 256), 256, 0, st>>>(gt_iv, n_gt, word_off, nframes, R, gmask);
        B200VAD_LAUNCH_CHECK();
    }
    if (n_pred > 0) {
        raster_intervals_kernel<<<(unsigned)((n_pred * 32 + 255) / 256), 256, 0, st>>>(pred_iv, n_pred, word_off, nframes, R, pmask);
        B200VAD_LAUNCH_CHECK();
    }
    if (total_words > 0) {
        int chunks = std::max(1, std::min(64, (max_words_per_rec_hint + 255) / 256));
        for (int r0 = 0; r0 < R; r0 += 65535) {
            const int rc = std::min(65535, R - r0);
            dim3 grid(chunks, rc);
            count_fa_md_kernel<<<grid, 256, 0, st>>>(gmask, pmask, word_off + r0, reinterpret_cast<unsigned long long*>(fa) + r0,
                                                     reinterpret_cast<unsigned long long*>(md) + r0);
            B200VAD_LAUNCH_CHECK();
        }
    }
    return B200VAD_OK;
}

// ---------------------------------------------------------------- long-form: centre-crop stitching
// prob: (W, Tw) per-window values; window w starts at global frame w * hop.  out: (L) stitched stream.
// Frame f belongs to window w = clamp((f - (Tw - hop) / 2) / hop, 0, W - 1) (shifted down while f falls outside it).
template <typename T>
__global__ void __launch_bounds__(256)
stitch_center_kernel(const T* __restrict__ prob, int W, int Tw, int hop, T* __restrict__ out, int64_t L, T fill) {
    const int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= L) return;
    const int margin = (Tw - hop) / 2;
    int64_t w = (f - margin) / hop;
    if (f < margin) w = 0;
    if (w > W - 1) w = W - 1;
    const int64_t k = f - w * hop;
    out[f] = (k >= 0 && k < Tw) ? prob[w * Tw + k] : fill;
}
int stitch_center_launch(const float* prob, int W, int Tw, int hop, float* out, int64_t L, cudaStream_t st) {
    if (L <= 0) return B200VAD_OK;
    stitch_center_kernel<float><<<(unsigned)((L + 255) / 256), 256, 0, st>>>(prob, W, Tw, hop, out, L, 0.f);
    B200VAD_LAUNCH_CHECK();
    return B200VAD_OK;
}

// ---------------------------------------------------------------- streaming: ring append + linearise
// ring: (S, 2 * Wn) double-write ring; chunk: (S, hop) new samples; pos = write index in [0, Wn) before the append.
// After the append the last Wn samples of stream s are ring[s][pos + hop .. pos + hop + Wn); they are copied to lin (S, Wn).
__global__ void __launch_bounds__(256)
stream_append_kernel(float* __restrict__ ring, const float* __restrict__ chunk, int S, int Wn, int hop, int pos) {
    const int s = blockIdx.y;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < hop; i += gridDim.x * blockDim.x) {
        const float v = chunk[(int64_t)s * hop + i];
        int p = pos + i;
        if (p >= Wn) p -= Wn;
        float* row = ring + (int64_t)s * 2 * Wn;
        row[p] = v;
        row[p + Wn] = v;
    }
}
__global__ void __launch_bounds__(256)
stream_linearise_kernel(const float* __restrict__ ring, float* __restrict__ lin, int S, int Wn, int start) {
    const int s = blockIdx.y;
    const float* src = ring + (int64_t)s * 2 * Wn + start;
    float* dst = lin + (int64_t)s * Wn;
    if (((Wn | start) & 3) == 0) {
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < Wn / 4; i += gridDim.x * blockDim.x)
            reinterpret_cast<float4*>(dst)[i] = __ldg(reinterpret_cast<const float4*>(src) + i);
    } else {   // SincNet hops (multiples of 270 samples) leave the window start off 16-byte boundaries
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < Wn; i += gridDim.x * blockDim.x) dst[i] = __ldg(src + i);
    }
}
// newest `nf` frames of every stream: prob (S, T) / dec (S, T) -> (S, nf)
__global__ void stream_newest_kernel(const float* __restrict__ prob, const uint8_t* __restrict__ dec, int S, int64_t T, int nf,
                                     float* __restrict__ prob_out, uint8_t* __restrict__ dec_out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= S * nf) return;
    const int s = i / nf, k = i - s * nf;
    const int64_t t = T - nf + k;
    prob_out[i] = prob[(int64_t)s * T + t];
    dec_out[i] = dec[(int64_t)s * T + t];
}

int stream_append_launch(float* ring, const float* chunk, float* lin, int S, int Wn, int hop, int pos, cudaStream_t st) {
    dim3 g1(std::max(1, (hop + 255) / 256), S);
    stream_append_kernel<<<g1, 256, 0, st>>>(ring, chunk, S, Wn, hop, pos);
    B200VAD_LAUNCH_CHECK();
    int start = pos + hop;
    if (start >= Wn) start -= Wn;
    dim3 g2(std::max(1, std::min(32, (Wn / 4 + 255) / 256)), S);
    stream_linearise_kernel<<<g2, 256, 0, st>>>(ring, lin, S, Wn, start);
    B200VAD_LAUNCH_CHECK();
    return B200VAD_OK;
}
int stream_newest_launch(const float* prob, const uint8_t* dec, int S, int64_t T, int nf, float* prob_out, uint8_t* dec_out,
                         cudaStream_t st) {
    stream_newest_kernel<<<(S * nf + 255) / 256, 256, 0, st>>>(prob, dec, S, T, nf, prob_out, dec_out);
    B200VAD_LAUNCH_CHECK();
    return B200VAD_OK;
}

// ---------------------------------------------------------------- synthetic corpus (BASELINE config 4)
// Deterministic per (seed, utterance id, sample index), independent of batching / sharding: 0.5 s segments that are
// either background noise or noise + an amplitude-modulated 3-harmonic voiced burst.  A 1000-hour corpus is generated
// batch by batch on the device instead of being held (230 GB) on the host.
__device__ __forceinline__ uint32_t mix32(uint64_t x) {
    x ^= x >> 33; x *= 0xff51afd7ed558ccdULL; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ULL; x ^= x >> 33;
    return (uint32_t)x;
}
__global__ void __launch_bounds__(256)
synth_corpus_kernel(float* __restrict__ out, int64_t utt0, int rows, int64_t N, uint64_t seed) {
    const int r = blockIdx.y;
    const uint64_t utt = (uint64_t)(utt0 + r);
    const uint64_t key = seed * 0x9E3779B97F4A7C15ULL + utt * 0xD1B54A32D192ED03ULL;
    const float f0 = 90.f + 160.f * (mix32(key ^ 0xF0F0) * (1.f / 4294967296.f));
    const float namp = exp10f(-3.f + (mix32(key ^ 0xA5A5) * (1.f / 4294967296.f)));
    for (int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t h = mix32(key + 0x632BE59BD9B4E019ULL * (uint64_t)(n + 1));
        // sum of four bytes: mean 510, sigma ~147.8 -> roughly normal
        const float g = ((float)((h & 255) + ((h >> 8) & 255) + ((h >> 16) & 255) + (h >> 24)) - 510.f) * (1.f / 147.8f);
        float x = namp * g;
        const int64_t segi = n / 8000;
        if (mix32(key ^ (0x5EED0000ULL + (uint64_t)segi)) & 1u) {
            const float t = (float)(n % 16000) * (1.f / 16000.f) + (float)((n / 16000) % 8);   // phase-continuous per 8 s
            const float w = 6.2831853f * f0 * t;
            const float am = 0.5f * (1.f + __sinf(6.2831853f * 3.f * t));
            x += 0.1f * am * (__sinf(w) + 0.5f * __sinf(2.f * w) + 0.3333333f * __sinf(3.f * w));
        }
        out[(int64_t)r * N + n] = x;
    }
}
int synth_corpus_launch(float* out, int64_t utt0, int rows, int64_t N, uint64_t seed, cudaStream_t st) {
    if (rows <= 0 || N <= 0) return B200VAD_OK;
    dim3 grid((unsigned)std::min<int64_t>((N + 255) / 256, 64), rows);
    synth_corpus_kernel<<<grid, 256, 0, st>>>(out, utt0, rows, N, seed);
    B200VAD_LAUNCH_CHECK();
    return B200VAD_OK;
}

}  // namespace b200vad
