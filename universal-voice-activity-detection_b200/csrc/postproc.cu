// Threshold + median smoothing + run-length segment extraction on the GPU.
//
// Replaces src/utils/helper.py:66-97 (torch.where(x < 0.5, 0, 1) -> .cpu() -> scipy
// medfilt(k) per row -> .to("cuda")) and the per-frame Python loop of
// src/scripts/predict.py:472-490.  On 0/1 data the zero-padded median of an odd window k
// is 1 iff the window sum >= (k+1)/2, so the filter is a sliding popcount: ballot words ->
// prefix sums in shared memory -> two lookups per frame.  HBM traffic: 4 B/frame in,
// 1 B (or 8 B for the reference's int64 view) out.
#include "kernels.cuh"

namespace b200vad {

constexpr int kMedTile = 2048;      // frames per CTA
constexpr int kMedMaxHalo = 512;    // supports kernel sizes up to 1025

// prob: [B][T] fp32.  out: [B][T] uint8 (elem=1) or int64 (elem=8).  NaN -> 1 (x < thr is false).
// With stream_off (B + 1 offsets), row b is the stream prob[stream_off[b], stream_off[b + 1]) instead, zero padded at its own
// edges, and T bounds the stream lengths (grid.x covers T); its decisions go to the same offsets of out.
__global__ void __launch_bounds__(256)
threshold_median_kernel(const float* __restrict__ prob, const int64_t* __restrict__ stream_off, int B, int64_t T, float thr, int half,
                        void* __restrict__ out, int elem, int32_t* __restrict__ near_count, float near_tol) {
    __shared__ int pre[kMedTile + 2 * kMedMaxHalo + 1];
    __shared__ int warp_tot[8];
    const int b = blockIdx.y;
    const int64_t t0 = (int64_t)blockIdx.x * kMedTile;
    const int64_t first = stream_off ? stream_off[b] : (int64_t)b * T;     // the row's first frame in prob and out
    if (stream_off) T = stream_off[b + 1] - first;
    if (t0 >= T) return;                            // the whole CTA: this stream is shorter than the longest one
    const int span = kMedTile + 2 * half;           // frames [t0 - half, t0 + tile + half)
    const float* row = prob + first;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int near = 0;
    // exclusive prefix sum of decisions over the span, 256 frames per round
    int carry = 0;
    for (int base = 0; base < span; base += 256) {
        int s = base + tid;
        int64_t t = t0 - half + s;
        int d = 0;
        if (s < span && t >= 0 && t < T) {
            float p = __ldg(row + t);
            d = (p < thr) ? 0 : 1;
            if (near_count && s >= half && s < half + kMedTile && fabsf(p - thr) <= near_tol) near++;
        }
        unsigned m = __ballot_sync(0xffffffffu, d);
        int incl = __popc(m & (0xffffffffu >> (31 - lane)));
        if (lane == 31) warp_tot[warp] = incl;
        __syncthreads();
        int off = carry;
#pragma unroll
        for (int w = 0; w < 8; ++w) {
            int v = warp_tot[w];
            if (w < warp) off += v;
            carry += v;
        }
        if (s < span) pre[s + 1] = off + incl;
        __syncthreads();
    }
    if (tid == 0) pre[0] = 0;
    __syncthreads();
    const int need = half + 1;                      // (k+1)/2 with k = 2*half+1
    for (int i = tid; i < kMedTile; i += 256) {
        int64_t t = t0 + i;
        if (t >= T) break;
        int sum = pre[i + 2 * half + 1] - pre[i];   // window [t-half, t+half]
        int v = sum >= need;
        if (elem == 1) reinterpret_cast<uint8_t*>(out)[first + t] = (uint8_t)v;
        else reinterpret_cast<int64_t*>(out)[first + t] = (int64_t)v;
    }
    if (near_count) {
        near = (int)warp_sum((float)near);
        if (lane == 0 && near) atomicAdd(near_count, near);
    }
}

int threshold_median_launch(const float* prob, int B, int64_t T, float thr, int kernel, void* out, int elem,
                            int32_t* near_count, float near_tol, cudaStream_t stream, const int64_t* stream_off) {
    if (B == 0 || T == 0) return B200VAD_OK;
    if (kernel < 1 || (kernel & 1) == 0 || kernel / 2 > kMedMaxHalo) {
        set_error("threshold_median: kernel size must be odd and <= %d", 2 * kMedMaxHalo + 1);
        return B200VAD_EINVAL;
    }
    int half = kernel / 2;
    dim3 grid((unsigned)((T + kMedTile - 1) / kMedTile), B);
    threshold_median_kernel<<<grid, 256, 0, stream>>>(prob, stream_off, B, T, thr, half, out, elem, near_count, near_tol);
    B200VAD_LAUNCH_CHECK();
    return B200VAD_OK;
}

// ---------------------------------------------------------------- run-length segments
// dec: flat uint8 stream; stream r = dec[offsets[r], offsets[r+1]).  A run of >= min_run
// consecutive non-zero frames yields (r, first, last_inclusive), frame indices relative to the
// stream start (predict.py:472-490 keeps a run iff round(end,2) - round(start,2) > 0, i.e.
// length >= 2).  Pass 1 counts per stream, an exclusive scan orders the output by (r, first),
// pass 2 writes.  One CTA per stream, 32 frames per thread-iteration via ballot.
template <bool WRITE>
__global__ void __launch_bounds__(256)
segments_kernel(const uint8_t* __restrict__ dec, const int64_t* __restrict__ offsets, int64_t uniform_T, int R, int min_run,
                int row_base, int32_t* __restrict__ counts, const int64_t* __restrict__ seg_off, int32_t* __restrict__ seg, int64_t cap) {
    const int r = blockIdx.x;
    const int64_t beg = offsets ? offsets[r] : (int64_t)r * uniform_T;
    const int64_t len = offsets ? offsets[r + 1] - beg : uniform_T;
    const uint8_t* d = dec + beg;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    __shared__ int wsum[8];
    __shared__ int s_carry;
    __shared__ int s_open_start;     // start frame of a run still open at the chunk boundary (or -1)
    if (tid == 0) { s_carry = 0; s_open_start = -1; }
    __syncthreads();
    int64_t out_base = WRITE ? seg_off[r] : 0;
    // every chunk = 256 frames, one frame per thread; runs are closed at their END frame:
    // an end at frame e (d[e]=1, d[e+1]=0 or e=len-1) emits (start, e) where start is found by a
    // backward scan limited to the chunk, falling back to the carried open start.
    for (int64_t base = 0; base < len; base += 256) {
        int64_t t = base + tid;
        int cur = (t < len) ? (d[t] != 0) : 0;
        int nxt = (t + 1 < len) ? (d[t + 1] != 0) : 0;
        unsigned m = __ballot_sync(0xffffffffu, cur);
        __shared__ unsigned words[8];
        if (lane == 0) words[warp] = m;
        __syncthreads();
        int is_end = cur && !nxt;
        int start = -1;
        int valid = 0;
        if (is_end) {
            // backward scan for the first zero before tid within this chunk
            int pos = tid;           // position in chunk
            int w = pos >> 5;
            unsigned inv = ~words[w] & (0xffffffffu >> (31 - (pos & 31)));   // zeros at or before pos in word
            int zero_at = -1;
            while (true) {
                if (inv) { zero_at = (w << 5) + 31 - __clz(inv); break; }
                if (--w < 0) break;
                inv = ~words[w];
            }
            int64_t st;
            if (zero_at >= 0) st = base + zero_at + 1;
            else st = (s_open_start >= 0) ? (int64_t)s_open_start : base;    // run spans the chunk start
            start = (int)st;
            valid = (t - st + 1) >= min_run;
        }
        unsigned vm = __ballot_sync(0xffffffffu, valid);
        int incl = __popc(vm & (0xffffffffu >> (31 - lane)));
        if (lane == 31) wsum[warp] = incl;
        __syncthreads();
        int off = s_carry, tot = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) {
            if (w < warp) off += wsum[w];
            tot += wsum[w];
        }
        if (WRITE && valid) {
            int64_t o = out_base + off + incl - 1;
            if (o < cap) {
                seg[o * 3 + 0] = r + row_base;
                seg[o * 3 + 1] = start;
                seg[o * 3 + 2] = (int)t;
            }
        }
        __syncthreads();
        if (tid == 255) {
            // s_open_start := start of the run still open at the end of this chunk (or -1)
            if (!cur) {
                s_open_start = -1;
            } else {
                int w = 7, zero_at = -1;
                unsigned inv = ~words[7];
                while (true) {
                    if (inv) { zero_at = (w << 5) + 31 - __clz(inv); break; }
                    if (--w < 0) break;
                    inv = ~words[w];
                }
                if (zero_at >= 0) s_open_start = (int)(base + zero_at + 1);
                else if (s_open_start < 0) s_open_start = (int)base;
            }
            s_carry += tot;
        }
        __syncthreads();
    }
    if (!WRITE && tid == 0) counts[r] = s_carry;
}

// exclusive scan of counts[R] -> seg_off[R+1] (int64); single CTA, R up to millions is fine (serial chunks)
__global__ void __launch_bounds__(1024) scan_counts_kernel(const int32_t* __restrict__ counts, int R, int64_t* __restrict__ seg_off) {
    __shared__ long long wtot[32];
    __shared__ long long carry;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) carry = 0;
    __syncthreads();
    for (int base = 0; base < R; base += 1024) {
        int i = base + tid;
        long long v = (i < R) ? counts[i] : 0;
        long long incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            long long n = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += n;
        }
        if (lane == 31) wtot[warp] = incl;
        __syncthreads();
        long long off = carry;
        for (int w = 0; w < warp; ++w) off += wtot[w];
        if (i < R) seg_off[i] = off + incl - v;
        __syncthreads();
        if (tid == 1023) carry = off + incl;
        __syncthreads();
    }
    if (tid == 0) seg_off[R] = carry;
}

int segments_launch(const uint8_t* dec, const int64_t* offsets, int64_t uniform_T, int R, int min_run, int row_base,
                    int32_t* counts, int64_t* seg_off, int32_t* seg, int64_t cap, cudaStream_t stream) {
    if (R == 0) return B200VAD_OK;
    segments_kernel<false><<<R, 256, 0, stream>>>(dec, offsets, uniform_T, R, min_run, row_base, counts, nullptr, nullptr, 0);
    B200VAD_LAUNCH_CHECK();
    scan_counts_kernel<<<1, 1024, 0, stream>>>(counts, R, seg_off);
    B200VAD_LAUNCH_CHECK();
    segments_kernel<true><<<R, 256, 0, stream>>>(dec, offsets, uniform_T, R, min_run, row_base, counts, seg_off, seg, cap);
    B200VAD_LAUNCH_CHECK();
    return B200VAD_OK;
}

// ---------------------------------------------------------------- binarization (onset / offset hysteresis, pads, min durations)
// pyannote's Binarize in the frame domain (include/b200vad.h states the contract).  Steps 2-4 of the contract collapse into one
// rule on the hysteresis output a[]: two consecutive regions [s1, e1), [s2, e2) belong to one group iff their gap
// s2 - e1 < G = pad_onset + pad_offset + max(min_off, 1) (padded gap below max(min_off, 1): they overlap, touch or the gap is
// filled).  A group [S, E) becomes [max(0, S - pad_onset), min(len, E + pad_offset)) and survives iff that is >= min_on
// frames long.  So a group is closed when the NEXT group starts (or at the end of the stream), and no pad or duration needs a
// halo: the kernel carries four numbers across chunks (hysteresis state, last region end, open group start, groups so far).
//
// One CTA per stream walks it in chunks of 2048 frames = 64 words of 32; every per-frame step is a ballot and every
// cross-word step is a 64-entry scan by warp 0, so a chunk costs a fixed handful of barriers whatever its content.
// Pass 1 counts, scan_counts_kernel orders the output by (r, s), pass 2 writes, binarize_raster_kernel fills dec from the
// triples (a padded group can reach any distance back or forth, so dec is written once all groups are known).
constexpr int kBinThreads = 256;
constexpr int kBinWords = 64;                       // words per chunk
constexpr int kBinChunk = 32 * kBinWords;           // frames per chunk
constexpr int kBinRounds = kBinChunk / kBinThreads; // frames per thread per chunk

// position of the last set bit of each of the 64 words before w, as an exclusive running "last" over the chunk (or `carry`);
// warp 0, lane l owns words l and l + 32.  pos(w) = the word's own last position or -1.
__device__ __forceinline__ void last_pos_scan(int lane, int64_t pos_lo, int64_t pos_hi, int64_t carry, int64_t* out /* [65] */) {
    int64_t v = pos_lo;                              // inclusive running max over words 0..l (positions increase with w)
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int64_t n = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v = max(v, n);
    }
    int64_t lo_incl = max(v, carry);
    int64_t lo_tot = __shfl_sync(0xffffffffu, lo_incl, 31);
    v = pos_hi;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int64_t n = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v = max(v, n);
    }
    int64_t hi_incl = max(v, lo_tot);
    int64_t lo_excl = __shfl_up_sync(0xffffffffu, lo_incl, 1);
    int64_t hi_excl = __shfl_up_sync(0xffffffffu, hi_incl, 1);
    out[lane] = lane ? lo_excl : carry;
    out[lane + 32] = lane ? hi_excl : lo_tot;
    if (lane == 31) out[64] = hi_incl;
}

template <bool WRITE>
__global__ void __launch_bounds__(kBinThreads)
binarize_kernel(const float* __restrict__ prob, const int64_t* __restrict__ offsets, int64_t uniform_T, b200vad_binarize_params p,
                int row_base, int32_t* __restrict__ counts, const int64_t* __restrict__ seg_off, int32_t* __restrict__ seg, int64_t cap) {
    const int r = blockIdx.x;
    const int64_t beg = offsets ? offsets[r] : (int64_t)r * uniform_T;
    const int64_t len = offsets ? offsets[r + 1] - beg : uniform_T;
    const float* x = prob + beg;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t gap_break = (int64_t)p.pad_onset + p.pad_offset + max(p.min_off, 1);
    __shared__ unsigned s1w[kBinWords], s0w[kBinWords], aw[kBinWords], stw[kBinWords], enw[kBinWords], gsw[kBinWords], emw[kBinWords];
    __shared__ int cin[kBinWords + 1];
    __shared__ int64_t last_end[kBinWords + 1], last_gs[kBinWords + 1];
    __shared__ int emit_off[kBinWords + 1];
    __shared__ int c_a;                // hysteresis state before the chunk
    __shared__ int64_t c_end, c_gs;    // last region end, start of the open group (-1: none)
    __shared__ int64_t c_count;        // surviving groups so far
    if (tid == 0) { c_a = 0; c_end = -1; c_gs = -1; c_count = 0; }
    __syncthreads();
    const int64_t out_base = WRITE ? seg_off[r] : 0;
    // a group [gs, ge) of raw frames -> 1 if it survives, with its padded, clipped bounds
    auto survive = [&](int64_t gs, int64_t ge, int64_t& a, int64_t& b) {
        a = gs - p.pad_onset;
        if (a < 0) a = 0;
        b = ge + p.pad_offset;
        if (b > len) b = len;
        return b - a >= p.min_on;
    };
    for (int64_t base = 0; base < len; base += kBinChunk) {
        // 1. the frames that set the state to 1 / to 0
#pragma unroll
        for (int k = 0; k < kBinRounds; ++k) {
            const int64_t t = base + k * kBinThreads + tid;
            const float v = t < len ? __ldg(x + t) : 0.f;
            const unsigned m1 = __ballot_sync(0xffffffffu, t < len && v > p.onset);
            const unsigned m0 = __ballot_sync(0xffffffffu, t < len && v < p.offset);
            if (lane == 0) { s1w[k * 8 + warp] = m1; s0w[k * 8 + warp] = m0; }
        }
        __syncthreads();
        // 2. hysteresis state entering every word: the value of the last setting frame before it
        if (warp == 0) {
            auto last_val = [&](int w) { unsigned s = s1w[w] | s0w[w]; return (int)((s1w[w] >> (31 - __clz(s))) & 1u); };
            const unsigned h_lo = __ballot_sync(0xffffffffu, (s1w[lane] | s0w[lane]) != 0);
            const unsigned h_hi = __ballot_sync(0xffffffffu, (s1w[lane + 32] | s0w[lane + 32]) != 0);
            const unsigned long long H = (unsigned long long)h_lo | ((unsigned long long)h_hi << 32);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int w = lane + 32 * h;
                const unsigned long long m = H & ((1ull << w) - 1ull);
                cin[w] = m ? last_val(63 - __clzll(m)) : c_a;
            }
            if (lane == 0) cin[kBinWords] = H ? last_val(63 - __clzll(H)) : c_a;
        }
        __syncthreads();
        // 3. a[] per frame: the last setting frame at or before it in the word, else the word's carry-in
#pragma unroll
        for (int k = 0; k < kBinRounds; ++k) {
            const int w = k * 8 + warp;
            const unsigned s = (s1w[w] | s0w[w]) & (0xffffffffu >> (31 - lane));
            const int a = s ? (int)((s1w[w] >> (31 - __clz(s))) & 1u) : cin[w];
            const unsigned m = __ballot_sync(0xffffffffu, a && base + k * kBinThreads + tid < len);
            if (lane == 0) aw[w] = m;
        }
        __syncthreads();
        // 4. region starts and ends (an end is the first 0 after a run; the end at len is the flush below); last end before each word
        if (warp == 0) {
            int64_t pos[2];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int w = lane + 32 * h;
                const unsigned prev = w ? aw[w - 1] >> 31 : (unsigned)c_a;
                const int64_t t0 = base + 32 * w;
                const unsigned valid = t0 >= len ? 0u : (len - t0 >= 32 ? 0xffffffffu : (1u << (len - t0)) - 1u);
                const unsigned shifted = (aw[w] << 1) | prev;
                stw[w] = aw[w] & ~shifted;
                enw[w] = ~aw[w] & shifted & valid;
                pos[h] = enw[w] ? t0 + 31 - __clz(enw[w]) : -1;
            }
            last_pos_scan(lane, pos[0], pos[1], c_end, last_end);
        }
        __syncthreads();
        // 5. group starts: the first region, or a region whose gap to the previous region end is >= gap_break
#pragma unroll
        for (int k = 0; k < kBinRounds; ++k) {
            const int w = k * 8 + warp;
            const int64_t t = base + k * kBinThreads + tid;
            int g = 0;
            if ((stw[w] >> lane) & 1u) {
                const unsigned below = enw[w] & ((1u << lane) - 1u);
                const int64_t pe = below ? base + 32 * w + 31 - __clz(below) : last_end[w];
                g = pe < 0 || t - pe >= gap_break;
            }
            const unsigned m = __ballot_sync(0xffffffffu, g);
            if (lane == 0) gsw[w] = m;
        }
        __syncthreads();
        if (warp == 0) {
            int64_t pos[2];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int w = lane + 32 * h;
                pos[h] = gsw[w] ? base + 32 * w + 31 - __clz(gsw[w]) : -1;
            }
            last_pos_scan(lane, pos[0], pos[1], c_gs, last_gs);
        }
        __syncthreads();
        // 6. every group start closes the group before it: [previous group start, last region end before this start)
        int64_t gs_prev[kBinRounds], ge_prev[kBinRounds];
#pragma unroll
        for (int k = 0; k < kBinRounds; ++k) {
            const int w = k * 8 + warp;
            int e = 0;
            gs_prev[k] = -1; ge_prev[k] = -1;
            if ((gsw[w] >> lane) & 1u) {
                const unsigned gb = gsw[w] & ((1u << lane) - 1u), eb = enw[w] & ((1u << lane) - 1u);
                gs_prev[k] = gb ? base + 32 * w + 31 - __clz(gb) : last_gs[w];
                ge_prev[k] = eb ? base + 32 * w + 31 - __clz(eb) : last_end[w];
                int64_t a, b;
                e = gs_prev[k] >= 0 && survive(gs_prev[k], ge_prev[k], a, b);
            }
            const unsigned m = __ballot_sync(0xffffffffu, e);
            if (lane == 0) emw[w] = m;
        }
        __syncthreads();
        if (warp == 0) {
            const int c_lo = __popc(emw[lane]), c_hi = __popc(emw[lane + 32]);
            int v = c_lo;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                int n = __shfl_up_sync(0xffffffffu, v, o);
                if (lane >= o) v += n;
            }
            const int lo_tot = __shfl_sync(0xffffffffu, v, 31);
            emit_off[lane] = v - c_lo;
            int u = c_hi;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                int n = __shfl_up_sync(0xffffffffu, u, o);
                if (lane >= o) u += n;
            }
            emit_off[lane + 32] = lo_tot + u - c_hi;
            if (lane == 31) emit_off[kBinWords] = lo_tot + u;
        }
        __syncthreads();
        if (WRITE) {
#pragma unroll
            for (int k = 0; k < kBinRounds; ++k) {
                const int w = k * 8 + warp;
                if ((emw[w] >> lane) & 1u) {
                    const int64_t o = out_base + c_count + emit_off[w] + __popc(emw[w] & ((1u << lane) - 1u));
                    int64_t a, b;
                    survive(gs_prev[k], ge_prev[k], a, b);
                    if (o < cap) {
                        seg[o * 3 + 0] = r + row_base;
                        seg[o * 3 + 1] = (int)a;
                        seg[o * 3 + 2] = (int)(b - 1);
                    }
                }
            }
        }
        __syncthreads();
        if (tid == 0) {
            c_a = cin[kBinWords];
            c_end = last_end[kBinWords];
            c_gs = last_gs[kBinWords];
            c_count += emit_off[kBinWords];
        }
        __syncthreads();
    }
    if (tid == 0) {
        // the last group ends at the last region end, or at len if a region is still open
        int64_t a, b;
        const int64_t ge = c_a ? len : c_end;
        const bool last = c_gs >= 0 && survive(c_gs, ge, a, b);
        if (!WRITE) {
            counts[r] = (int32_t)(c_count + last);
        } else if (last) {
            const int64_t o = out_base + c_count;
            if (o < cap) {
                seg[o * 3 + 0] = r + row_base;
                seg[o * 3 + 1] = (int)a;
                seg[o * 3 + 2] = (int)(b - 1);
            }
        }
    }
}

// dec[i] = 1 iff frame i lies in one of its stream's (disjoint, sorted) written groups: a binary search per frame
__global__ void __launch_bounds__(256)
binarize_raster_kernel(const int64_t* __restrict__ offsets, int64_t uniform_T, int R, int64_t total, const int64_t* __restrict__ seg_off,
                       const int32_t* __restrict__ seg, int64_t cap, uint8_t* __restrict__ dec) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    int r;
    int64_t t;
    if (offsets) {
        // the last stream starting at or before i (skips empty streams); frames outside [offsets[0], offsets[R]) are no stream's
        if (i < offsets[0] || i >= offsets[R]) { dec[i] = 0; return; }
        int lo = 0, hi = R - 1;
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (offsets[mid] <= i) lo = mid; else hi = mid - 1;
        }
        r = lo;
        t = i - offsets[r];
    } else {
        r = (int)(i / uniform_T);
        t = i - (int64_t)r * uniform_T;
    }
    int64_t lo = seg_off[r], hi = min(seg_off[r + 1], cap) - 1;   // last group with start <= t
    int64_t found = -1;
    while (lo <= hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (seg[mid * 3 + 1] <= t) { found = mid; lo = mid + 1; } else hi = mid - 1;
    }
    dec[i] = found >= 0 && t <= seg[found * 3 + 2];
}

int binarize_launch(const float* prob, const int64_t* offsets, int64_t T, int R, const b200vad_binarize_params& p, int row_base,
                    uint8_t* dec, int32_t* counts, int64_t* seg_off, int32_t* seg, int64_t cap, cudaStream_t stream) {
    if (R == 0) return B200VAD_OK;
    const int64_t uniform_T = offsets ? 0 : T;
    binarize_kernel<false><<<R, kBinThreads, 0, stream>>>(prob, offsets, uniform_T, p, row_base, counts, nullptr, nullptr, 0);
    B200VAD_LAUNCH_CHECK();
    scan_counts_kernel<<<1, 1024, 0, stream>>>(counts, R, seg_off);
    B200VAD_LAUNCH_CHECK();
    binarize_kernel<true><<<R, kBinThreads, 0, stream>>>(prob, offsets, uniform_T, p, row_base, counts, seg_off, seg, cap);
    B200VAD_LAUNCH_CHECK();
    const int64_t total = offsets ? T : (int64_t)R * T;
    if (total > 0) {
        binarize_raster_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(offsets, uniform_T, R, total, seg_off, seg, cap, dec);
        B200VAD_LAUNCH_CHECK();
    }
    return B200VAD_OK;
}


// ---------------------------------------------------------------- streaming speech events (include/b200vad.h states the contract)
// One warp per stream walks its new frames 32 at a time, with the group rule of binarize_kernel.  Per word, every lane owns one
// frame and finds from ballots of the word and the carried state: the hysteresis value (last setting frame at or before it),
// region starts and ends, the last region end at or before it, whether a rise starts a new group (no group open, or >= gap_break
// frames after that end), whether its frame closes the open group (a[t] = 0 and t = last end + gap_break - 1), the group in
// effect during its frame and that group's start test.  A start is the first frame of a group whose test passes; an end is a
// close whose test passes.  So a word costs a fixed handful of ballots and the events come out compacted, in frame order.
constexpr int kEvWarps = 4;

__global__ void __launch_bounds__(32 * kEvWarps)
regions_step_kernel(const float* __restrict__ prob, int S, int nf, int64_t row_stride, b200vad_binarize_params p,
                    int64_t* __restrict__ state, const uint8_t* __restrict__ flush, int64_t* __restrict__ ev,
                    int32_t* __restrict__ ev_counts, int64_t cap) {
    const int r = blockIdx.x * kEvWarps + (threadIdx.x >> 5);
    if (r >= S) return;
    const int lane = threadIdx.x & 31;
    const unsigned lt = (1u << lane) - 1u, le = lt | (1u << lane);
    const int64_t gap_break = (int64_t)p.pad_onset + p.pad_offset + max(p.min_off, 1);
    int64_t* st = state + (int64_t)r * 5;
    int h = (int)st[0], status = (int)st[3];
    int64_t last_end = st[1], gs = st[2];
    const int64_t len = st[4];
    const float* x = prob + (int64_t)r * row_stride;
    int64_t* out = ev + (int64_t)r * cap * 2;
    int64_t n = 0;
    auto last = [](unsigned m) { return 31 - __clz(m); };
    for (int base = 0; base < nf; base += 32) {
        const int nv = min(32, nf - base);
        const bool valid = lane < nv;
        const unsigned vm = nv == 32 ? 0xffffffffu : (1u << nv) - 1u;
        const int64_t t0 = len + base, t = t0 + lane;
        const float v = valid ? __ldg(x + base + lane) : 0.f;
        const unsigned m1 = __ballot_sync(0xffffffffu, valid && v > p.onset);
        const unsigned m0 = __ballot_sync(0xffffffffu, valid && v < p.offset);
        const unsigned sm = (m1 | m0) & le;
        const int a = sm ? (int)((m1 >> last(sm)) & 1u) : h;
        const unsigned A = __ballot_sync(0xffffffffu, a) & vm;
        const unsigned shifted = (A << 1) | (unsigned)h;
        const unsigned rise = A & ~shifted, fall = ~A & shifted & vm;
        // last region end before / at or before t; the carried one counts only while its group is open (-1: none)
        const int64_t pe_carry = status ? last_end : -1;
        const int64_t pe_lt = (fall & lt) ? t0 + last(fall & lt) : pe_carry;
        const int64_t pe_le = (fall & le) ? t0 + last(fall & le) : pe_carry;
        const bool g = valid && ((rise >> lane) & 1u) && (pe_lt < 0 || t - pe_lt >= gap_break);
        const bool c = valid && !a && pe_le >= 0 && t - pe_le + 1 == gap_break;
        const unsigned G = __ballot_sync(0xffffffffu, g), C = __ballot_sync(0xffffffffu, c);
        // the group open during frame t: the latest of a group start at or before t and a close before t decides
        const unsigned gle = G & le, clt = C & lt;
        const bool open = valid && (gle ? (!clt || last(gle) > last(clt)) : (!clt && status != 0));
        const int64_t gst = gle ? t0 + last(gle) : gs;
        const int64_t s = max(gst - (int64_t)p.pad_onset, (int64_t)0);
        bool pass = false;
        if (open) {
            const int64_t ge = a ? t + 1 : pe_le;
            pass = min(t + 1, ge + (int64_t)p.pad_offset) - s >= (int64_t)p.min_on;
        }
        const unsigned P = __ballot_sync(0xffffffffu, pass);
        const bool passed_before = lane ? ((P >> (lane - 1)) & 1u) : status == 2;
        const bool start = pass && (g || !passed_before);
        const bool end = c && pass;
        const unsigned E = __ballot_sync(0xffffffffu, start || end);
        if (start || end) {
            const int64_t o = n + __popc(E & lt);
            if (o < cap) {
                out[2 * o] = start ? s : pe_le + p.pad_offset;
                out[2 * o + 1] = start;
            }
        }
        n += __popc(E);
        const int L = nv - 1;           // the state after the word is the one after its last frame
        h = __shfl_sync(0xffffffffu, a, L);
        last_end = __shfl_sync(0xffffffffu, pe_le, L);
        gs = __shfl_sync(0xffffffffu, gst, L);
        status = __shfl_sync(0xffffffffu, open && !c ? (pass ? 2 : 1) : 0, L);
    }
    if (lane != 0) return;
    if (flush && flush[r]) {
        // end of stream: only a group whose start was emitted survives (the start test at the last frame is the survival test)
        if (status == 2) {
            const int64_t T = len + nf;
            const int64_t e = min(T, (h ? T : last_end) + (int64_t)p.pad_offset);
            if (n < cap) { out[2 * n] = e; out[2 * n + 1] = 0; }
            ++n;
        }
        st[0] = st[1] = st[2] = st[3] = st[4] = 0;
    } else {
        st[0] = h; st[1] = last_end; st[2] = gs; st[3] = status; st[4] = len + nf;
    }
    ev_counts[r] = (int32_t)n;
}

int regions_step_launch(const float* prob, int S, int nf, int64_t row_stride, const b200vad_binarize_params& p, int64_t* state,
                        const uint8_t* flush, int64_t* ev, int32_t* ev_counts, int64_t cap, cudaStream_t stream) {
    if (S == 0) return B200VAD_OK;
    regions_step_kernel<<<(S + kEvWarps - 1) / kEvWarps, 32 * kEvWarps, 0, stream>>>(prob, S, nf, row_stride, p, state, flush, ev,
                                                                                     ev_counts, cap);
    B200VAD_LAUNCH_CHECK();
    return B200VAD_OK;
}

}  // namespace b200vad
