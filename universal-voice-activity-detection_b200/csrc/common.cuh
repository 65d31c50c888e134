// Shared device/host helpers for the b200vad kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>

#define B200VAD_OK 0
#define B200VAD_EINVAL (-1)
#define B200VAD_ECUDA (-2)
#define B200VAD_ENOMEM (-3)
#define B200VAD_ESTATE (-4)

namespace b200vad {

void set_error(const char* fmt, ...);
void count_launch();                       // bumps the process-wide kernel-launch counter
// live timing of the hot kernels (bench.py roofline): when enabled, every launch of kind
// 0 = LSTM recurrence, 1 = input-projection GEMM, 2 = head GEMMs / warp-MMA GEMMs, 3 = fbank
// is bracketed by CUDA events on its own stream
// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) once per (kernel, device); thread safe.  Returns a B200VAD_* code.
int set_max_dynamic_smem(const void* func, int bytes);
void prof_begin(int kind, cudaStream_t st);
void prof_end(int kind, cudaStream_t st);

#define B200VAD_CHECK_ARG(cond, msg)                                   \
    do {                                                               \
        if (!(cond)) {                                                 \
            b200vad::set_error("%s: invalid argument: %s", __func__, msg); \
            return B200VAD_EINVAL;                                     \
        }                                                              \
    } while (0)

#define B200VAD_CUDA(call)                                             \
    do {                                                               \
        cudaError_t e__ = (call);                                      \
        if (e__ != cudaSuccess) {                                      \
            b200vad::set_error("%s: %s failed: %s", __func__, #call, cudaGetErrorString(e__)); \
            return B200VAD_ECUDA;                                      \
        }                                                              \
    } while (0)

#define B200VAD_LAUNCH_CHECK()                                         \
    do {                                                               \
        cudaError_t e__ = cudaGetLastError();                          \
        if (e__ != cudaSuccess) {                                      \
            b200vad::set_error("%s: kernel launch failed: %s", __func__, cudaGetErrorString(e__)); \
            return B200VAD_ECUDA;                                      \
        }                                                              \
        b200vad::count_launch();                                       \
    } while (0)

// model / feature constants (reference: lhotse FbankConfig defaults; PyanNet2.py:60-67)
constexpr int kFrameLen = 400;
constexpr int kFrameShift = 160;
constexpr int kFftLen = 512;
constexpr int kNumMel = 80;
constexpr int kPadLeft = 120;
constexpr int kHidden = 128;
constexpr int kGates = 4 * kHidden;
constexpr float kLogEpsilon = -23.025850929940457f;   // lhotse LOG_EPSILON (feature pad value)
constexpr float kEpsilon = 1.1920928955078125e-07f;    // torch.finfo(float).eps

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ float fast_ex2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float fast_rcp(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// sigmoid / tanh from one ex2 + one rcp each (~2 ulp); arguments clamped so the
// exponential never overflows (sigmoid(+-30), tanh(+-15) are already 1 in fp32).
__device__ __forceinline__ float sigmoid_acc(float x) {
    x = fminf(fmaxf(x, -30.f), 30.f);
    return fast_rcp(1.f + fast_ex2(-1.4426950408889634f * x));
}
__device__ __forceinline__ float tanh_acc(float x) {
    x = fminf(fmaxf(x, -15.f), 15.f);
    float e = fast_ex2(2.8853900817779268f * x);   // exp(2x)
    return 1.f - 2.f * fast_rcp(e + 1.f);
}

// The packed LSTM weights (W_ih, W_hh, b_ih + b_hh) carry the exponent scaling of the gate non-linearities:
// rows of the i, f, o gates are multiplied by -log2(e), rows of the g gate by 2*log2(e), so that a gate
// pre-activation z arrives as the argument of ex2:  sigmoid(x) = 1 / (1 + 2^z),  tanh(x) = (2^z - 1) / (2^z + 1).
// This removes one multiply per gate and cell from the recurrence's pointwise loop.
constexpr float kLog2e = 1.4426950408889634f;
__host__ __device__ __forceinline__ float lstm_gate_scale(int row) {
    const int gate = (row % kGates) / kHidden;
    return gate == 2 ? 2.f * kLog2e : -kLog2e;
}
// z = -log2(e) * x  ->  sigmoid(x);  z = 2*log2(e) * x  ->  tanh(x)   (clamped so that 2^z stays finite)
__device__ __forceinline__ float sigmoid_pre(float z) {
    return fast_rcp(1.f + fast_ex2(fminf(fmaxf(z, -43.f), 43.f)));
}
__device__ __forceinline__ float tanh_pre(float z) {
    float e = fast_ex2(fminf(fmaxf(z, -43.f), 43.f));
    return 1.f - 2.f * fast_rcp(e + 1.f);
}

// ---- packed fp32 pairs (sm_100 FADD2 / FMUL2 / FFMA2): two columns of the recurrence per issue slot ----
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float a, float b) {
    f32x2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
    return r;
}
__device__ __forceinline__ void unpack2(f32x2 v, float& a, float& b) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v));
}
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) {
    f32x2 d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) {
    f32x2 d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
    f32x2 d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
// elementwise 2^min(z, 29)
__device__ __forceinline__ f32x2 ex2_clamped2(f32x2 z) {
    float a, b;
    unpack2(z, a, b);
    return pack2(fast_ex2(fminf(a, 29.f)), fast_ex2(fminf(b, 29.f)));
}
__device__ __forceinline__ f32x2 rcp2(f32x2 z) {
    float a, b;
    unpack2(z, a, b);
    return pack2(fast_rcp(a), fast_rcp(b));
}

// 1 / x for x >= 1 (finite) on the FMA pipe: exponent-flip seed (max error 12 %) + two cubic (Householder) refinements
// y <- y (1 + e + e^2), e = 1 - x y: error 0.12 -> 2e-3 -> 8e-9.  Trades 2 MUFU.RCP per pair for 9 FMA-pipe / ALU issues.
__device__ __forceinline__ f32x2 rcp2_fma(f32x2 x) {
    float a, b;
    unpack2(x, a, b);
    f32x2 y = pack2(__int_as_float(0x7EF311C7 - __float_as_int(a)), __int_as_float(0x7EF311C7 - __float_as_int(b)));
    const f32x2 nx = mul2(x, pack2(-1.f, -1.f)), one = pack2(1.f, 1.f);
#pragma unroll
    for (int it = 0; it < 2; ++it) {
        const f32x2 e = fma2(nx, y, one);
        y = fma2(y, fma2(e, e, e), y);
    }
    return y;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---- legacy warp MMA helpers (m16n8k16, fp16 x fp16 -> fp32) ----
__device__ __forceinline__ void mma_16816(float (&c)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}
__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], uint32_t addr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];\n"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldmatrix_x2(uint32_t (&r)[2], uint32_t addr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x2.shared.b16 {%0,%1}, [%2];\n"
                 : "=r"(r[0]), "=r"(r[1]) : "r"(addr));
}

// fp32 -> (hi, lo) fp16 pair with hi + lo ~= x to ~22 bits
// two fp16 planes that sum to x: first = fp16(s1 * x), second = fp16(x - first).  s1 = 1: the hi / lo split; s1 = 1 - 2^-6:
// the scaled split of the 2-product GEMMs (gemm_tc.cu)
__device__ __forceinline__ void split_scaled_f16(float x, float s1, __half& a, __half& b) {
    a = __float2half_rn(x * s1);
    b = __float2half_rn(x - __half2float(a));
}
// split_scaled_f16 of two values at once (x in the low halves): the same operations and roundings, packed conversions
__device__ __forceinline__ void split_scaled_f16x2(float x, float y, float s1, uint32_t& a, uint32_t& b) {
    const __half2 a2 = __floats2half2_rn(x * s1, y * s1);
    const float2 af = __half22float2(a2);
    const __half2 b2 = __floats2half2_rn(x - af.x, y - af.y);
    a = *reinterpret_cast<const uint32_t*>(&a2);
    b = *reinterpret_cast<const uint32_t*>(&b2);
}
// Order-independent accumulation of InstanceNorm partial sums with atomicAdd(double): every partial is rounded to a multiple of
// 2^-BITS, so the additions are exact (no rounding, hence no dependence on the order in which CTAs arrive) as long as the running
// sum stays below 2^(53 - BITS); beyond that it degrades to ordinary double rounding (still accurate, no longer order-independent).
// BITS = 32: quantum 2.3e-10 -- below the fp32 rounding of any partial above 4e-3 and negligible against InstanceNorm's eps = 1e-5
// for smaller ones (2^-16 was measurably too coarse: 3e-3 on the SincNet output of a 2000-sample input) --, exact up to sums of 2e6.
template <int BITS>
__device__ __forceinline__ double exact_partial(double x) {
    return rint(x * (double)(1ull << BITS)) * (1.0 / (double)(1ull << BITS));
}
__device__ __forceinline__ void split_f16(float x, __half& hi, __half& lo) {
    hi = __float2half_rn(x);
    lo = __float2half_rn(x - __half2float(hi));
}

}  // namespace b200vad
