// fg_math.cuh -- precision policy + counter-based RNG for the MPE step kernels (sm_100a).
//
// Ops<float>  : fp32 arithmetic, FMA contraction allowed, IEEE div/sqrt (no --use_fast_math).
// Ops<double> : fp64 arithmetic written with the explicit round-to-nearest intrinsics so nvcc can
//               never contract a*b+c into an FMA -- the fp64 build reproduces the reference's
//               numpy evaluation order (formation_gym/core.py:304-318,268-277) to the last bit
//               wherever CUDA's exp/log1p agree with glibc's.
//               np.linalg.norm of a 2-vector is sqrt(ddot) and the reference's BLAS contracts the
//               dot into fma(y,y,x*x) (see oracle/mpe_oracle.py norm2) -> Ops<double>::norm2.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace fg {

template <typename T> struct Ops;

template <> struct Ops<float> {
    typedef float2 R2;
    typedef unsigned int Bits;
    static __device__ __forceinline__ float add(float a, float b) { return a + b; }
    static __device__ __forceinline__ float sub(float a, float b) { return a - b; }
    static __device__ __forceinline__ float mul(float a, float b) { return a * b; }
    static __device__ __forceinline__ float div(float a, float b) { return a / b; }
    static __device__ __forceinline__ float sqrt_(float a) { return sqrtf(a); }
    static __device__ __forceinline__ float exp_(float a) { return expf(a); }
    static __device__ __forceinline__ float log1p_(float a) { return log1pf(a); }
    static __device__ __forceinline__ float log_(float a) { return logf(a); }
    static __device__ __forceinline__ float asin_(float a) { return asinf(a); }
    static __device__ __forceinline__ void sincos_(float a, float* s, float* c) { sincosf(a, s, c); }
    static __device__ __forceinline__ float sq2(float x, float y) { return x * x + y * y; }
    static __device__ __forceinline__ float norm2(float x, float y) { return sqrtf(x * x + y * y); }
    // the argument of norm2's square root: min_k norm2(v_k) == sqrt_(min_k norm2sq(v_k)) exactly (sqrt is monotonic and
    // correctly rounded), which replaces k square roots by one
    static __device__ __forceinline__ float norm2sq(float x, float y) { return x * x + y * y; }
    // Ordering key of a 2-vector's length for argsort / argmin decisions: the squared length (sqrt is
    // monotonic, so the order is the same except for sub-ulp ties the fp32 build cannot reproduce anyway).
    static __device__ __forceinline__ float lenkey(float x, float y) { return x * x + y * y; }
    // x / n for a small integer count n: multiply by the reciprocal (<= 1 ulp; the fp64 build divides).
    static __device__ __forceinline__ float div_count(float x, int n) { return x * (1.0f / (float)n); }
    static __device__ __forceinline__ Bits bits(float a) { return __float_as_uint(a); }
    static __device__ __forceinline__ float from_bits(Bits b) { return __uint_as_float(b); }
    static __device__ __forceinline__ R2 make(float x, float y) { return make_float2(x, y); }
    static __device__ __forceinline__ void stcs(R2* p, R2 v) { __stcs(p, v); }   // st.global.cs (streaming)
};

template <> struct Ops<double> {
    typedef double2 R2;
    typedef unsigned long long Bits;
    static __device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
    static __device__ __forceinline__ double sub(double a, double b) { return __dsub_rn(a, b); }
    static __device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
    static __device__ __forceinline__ double div(double a, double b) { return __ddiv_rn(a, b); }
    static __device__ __forceinline__ double sqrt_(double a) { return __dsqrt_rn(a); }
    static __device__ __forceinline__ double exp_(double a) { return exp(a); }
    static __device__ __forceinline__ double log1p_(double a) { return log1p(a); }
    static __device__ __forceinline__ double log_(double a) { return log(a); }
    static __device__ __forceinline__ double asin_(double a) { return asin(a); }
    static __device__ __forceinline__ void sincos_(double a, double* s, double* c) { sincos(a, s, c); }
    // np.square(x)+np.square(y) / scipy's running sum: two rounded products, one rounded add
    static __device__ __forceinline__ double sq2(double x, double y) {
        return __dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y));
    }
    // np.linalg.norm([x, y]) = sqrt(ddot) with the BLAS tail loop contracted to an FMA
    static __device__ __forceinline__ double norm2(double x, double y) {
        return __dsqrt_rn(__fma_rn(y, y, __dmul_rn(x, x)));
    }
    static __device__ __forceinline__ double norm2sq(double x, double y) { return __fma_rn(y, y, __dmul_rn(x, x)); }
    static __device__ __forceinline__ double lenkey(double x, double y) { return norm2(x, y); }   // as np.linalg.norm
    static __device__ __forceinline__ double div_count(double x, int n) { return __ddiv_rn(x, (double)n); }
    static __device__ __forceinline__ Bits bits(double a) { return (Bits)__double_as_longlong(a); }
    static __device__ __forceinline__ double from_bits(Bits b) { return __longlong_as_double((long long)b); }
    static __device__ __forceinline__ R2 make(double x, double y) { return make_double2(x, y); }
    static __device__ __forceinline__ void stcs(R2* p, R2 v) { __stcs(p, v); }
};

// ---- Philox4x32-10 (Salmon et al., SC'11).  counter = (env, agent, tick, purpose), key = seed ----
struct U4 { uint32_t x, y, z, w; };

enum Purpose : uint32_t {
    kResetAgent = 0,     // .xy -> agent position         (formation_hd_env.py:81)
    kResetLandmark = 1,  // .xy -> landmark position      (formation_hd_env.py:89)
    kResetIdealVel = 2,  // .xy -> ideal velocity         (formation_hd_env.py:95)
    kUNoise = 3,         // Box-Muller pair -> motor noise (core.py:232-233)
    kCNoise = 4,         // Box-Muller pair -> comm noise  (core.py:284-285)
    kAction = 5,         // .xy -> random-policy action    (test.py:20)
    kResetTarget = 6     // .x  -> task of a target bank (fg_targets), umulhi(x, K); agent = 0
};

__host__ __device__ __forceinline__ void philox_mulhilo(uint32_t a, uint32_t b, uint32_t* hi, uint32_t* lo) {
#ifdef __CUDA_ARCH__
    *lo = a * b;
    *hi = __umulhi(a, b);
#else
    uint64_t p = (uint64_t)a * (uint64_t)b;
    *lo = (uint32_t)p;
    *hi = (uint32_t)(p >> 32);
#endif
}

__host__ __device__ __forceinline__ U4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                     uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0, lo0, hi1, lo1;
        philox_mulhilo(0xD2511F53u, c0, &hi0, &lo0);
        philox_mulhilo(0xCD9E8D57u, c2, &hi1, &lo1);
        uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    U4 out; out.x = c0; out.y = c1; out.z = c2; out.w = c3;
    return out;
}

__device__ __forceinline__ U4 philox(uint64_t seed, uint32_t env, uint32_t agent, uint32_t tick, uint32_t purpose) {
    return philox4x32_10(env, agent, tick, purpose, (uint32_t)seed, (uint32_t)(seed >> 32));
}

// U(-1,1) on a 24-bit lattice: (x >> 8) * 2^-23 - 1.  Exact in fp32 AND fp64, so both builds draw
// bit-identical reset states and actions (np.random.uniform(-1, +1): statistical parity only).
template <typename T> __device__ __forceinline__ T uniform_pm1(uint32_t x) {
    return (T)(x >> 8) * (T)(1.0 / 8388608.0) - (T)1.0;
}

// two N(0,1) draws by Box-Muller from two 32-bit words (np.random.randn: statistical parity only)
template <typename T> __device__ __forceinline__ void normal_pair(uint32_t a, uint32_t b, T* n0, T* n1) {
    T u1 = ((T)(a >> 8) + (T)1.0) * (T)(1.0 / 16777216.0);          // (0,1]
    T u2 = (T)(b >> 8) * (T)(1.0 / 16777216.0);                     // [0,1)
    T r = Ops<T>::sqrt_((T)-2.0 * Ops<T>::log_(u1));
    T s, c;
    Ops<T>::sincos_((T)6.283185307179586476925286766559 * u2, &s, &c);
    *n0 = r * c;
    *n1 = r * s;
}
// fp32 build: the draws are noise on a 24-bit lattice -- parity with np.random.randn is statistical only -- so the hardware
// approximations (MUFU.LG2 / MUFU.SIN / MUFU.COS: ~2^-21 absolute on [0, 2 pi)) replace the ~60-instruction IEEE logf /
// sincosf sequences on the step path (u_noise = 0.1 at N = 9: 57.2 -> see DESIGN.md).  The fp64 build keeps libm.
template <> __device__ __forceinline__ void normal_pair<float>(uint32_t a, uint32_t b, float* n0, float* n1) {
    float u1 = ((float)(a >> 8) + 1.0f) * (1.0f / 16777216.0f);     // (0,1]
    float u2 = (float)(b >> 8) * (1.0f / 16777216.0f);              // [0,1)
    float r = sqrtf(-2.0f * __logf(u1));
    float s, c;
    __sincosf(6.283185307179586f * u2, &s, &c);
    *n0 = r * c;
    *n1 = r * s;
}

// q / d for q*d < 2^32 with magic = floor(2^32 / d) + 1 (exact; see DESIGN.md "index decode")
__device__ __forceinline__ uint32_t fastdiv(uint32_t q, uint32_t magic) { return magic ? __umulhi(q, magic) : q; }

}  // namespace fg
