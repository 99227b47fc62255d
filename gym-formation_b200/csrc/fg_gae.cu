// fg_gae.cu -- generalized advantage estimation (Schulman et al. 2016) over an on-policy rollout, on the device
// (sm_100a), with time-limit truncations bootstrapped from the value of the state the episode ended in.
//
// Layouts (include/formation_gym_b200.h fg_gae), M = E*N columns, column c = e*N + n: reward / adv / ret / final_value
// [T, E, N], value [T+1, E, N], done [T, E] uint8.  One thread owns one column and walks t = T-1 .. 0; warps are
// coalesced over c.  Every operation is a separately rounded intrinsic, so nvcc cannot contract a multiply-add and a
// numpy loop in the same dtype reproduces adv / ret bit for bit (DESIGN.md 3.3g).
#include <stdint.h>
#include <cmath>

#include "fg_host.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kAhead = 8;                                     // rollout steps whose loads are issued before their math
constexpr long long kMaxElems = 1ll << 48;                    // T*E*N: (T+1)*M*8 bytes stays far below 2^63

bool aligned(const void* p, size_t a) { return ((uintptr_t)p % a) == 0; }

template <typename T> struct Rn;
template <> struct Rn<float> {
    static __device__ __forceinline__ float mul(float a, float b) { return __fmul_rn(a, b); }
    static __device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
    static __device__ __forceinline__ float sub(float a, float b) { return __fsub_rn(a, b); }
};
template <> struct Rn<double> {
    static __device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
    static __device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
    static __device__ __forceinline__ double sub(double a, double b) { return __dsub_rn(a, b); }
};

// Each array element is touched once, so loads and stores are streaming (evict-first).  The loads of kAhead steps
// are issued before the recurrence consumes them: they depend on t only, never on `a`.
template <typename T>
__global__ void __launch_bounds__(kThreads) k_gae(const T* __restrict__ reward, const T* __restrict__ value,
                                                  const T* __restrict__ final_value, const uint8_t* __restrict__ done,
                                                  T* __restrict__ adv, T* __restrict__ ret, int T_, long long E, int N,
                                                  T g, T gl) {
    using R = Rn<T>;
    const long long M = E * N, stride = (long long)gridDim.x * blockDim.x;
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < M; c += stride) {
        const long long e = c / N;
        T a = T(0);
        T v_next = __ldcs(value + (long long)T_ * M + c);      // V(s_T) of the rollout's last state
        for (int t0 = T_ - 1; t0 >= 0; t0 -= kAhead) {
            T r[kAhead], v[kAhead], f[kAhead];
            bool d[kAhead];
#pragma unroll
            for (int k = 0; k < kAhead; ++k) {
                const int t = t0 - k;
                if (t >= 0) {
                    const long long i = (long long)t * M + c;
                    d[k] = __ldcs(done + (long long)t * E + e) != 0;
                    r[k] = __ldcs(reward + i);
                    v[k] = __ldcs(value + i);
                }
            }
#pragma unroll
            for (int k = 0; k < kAhead; ++k) {                 // (after all of the above: these wait for done)
                const int t = t0 - k;
                f[k] = T(0);
                if (t >= 0 && d[k] && final_value) f[k] = __ldcs(final_value + (long long)t * M + c);
            }
#pragma unroll
            for (int k = 0; k < kAhead; ++k) {
                const int t = t0 - k;
                if (t >= 0) {
                    const long long i = (long long)t * M + c;
                    const T nv = d[k] ? f[k] : v_next;         // a select: value[t+1] after a done is never used
                    const T delta = R::sub(R::add(r[k], R::mul(g, nv)), v[k]);
                    a = d[k] ? delta : R::add(delta, R::mul(gl, a));
                    __stcs(adv + i, a);
                    __stcs(ret + i, R::add(a, v[k]));
                    v_next = v[k];
                }
            }
        }
    }
}

template <typename T>
int gae_impl(const void* reward, const void* value, const void* final_value, const uint8_t* done, void* adv,
             void* ret, int T_, long long E, int N, double gamma, double lambda, void* stream, const char* who) {
    NvtxRange nvtx_(who);
    if (!reward || !value || !done || !adv || !ret)
        return fail(FG_ERR_ARG, "%s: reward / value / done / adv / ret must be non-null", who);
    if (T_ < 1) return fail(FG_ERR_ARG, "%s: T must be >= 1", who);
    if (E < 1) return fail(FG_ERR_ARG, "%s: E must be >= 1", who);
    if (N < 1 || N > FG_MAX_AGENTS) return fail(FG_ERR_ARG, "%s: N must be in [1, FG_MAX_AGENTS=256]", who);
    if (E > kMaxElems / ((long long)T_ * N)) return fail(FG_ERR_ARG, "%s: T * E * N must be <= 2^48", who);
    if (!std::isfinite(gamma) || gamma < 0.0 || gamma > 1.0)
        return fail(FG_ERR_ARG, "%s: gamma must be finite and in [0, 1]", who);
    if (!std::isfinite(lambda) || lambda < 0.0 || lambda > 1.0)
        return fail(FG_ERR_ARG, "%s: lambda must be finite and in [0, 1]", who);
    if (!aligned(reward, sizeof(T)) || !aligned(value, sizeof(T)) || !aligned(final_value, sizeof(T)) ||
        !aligned(adv, sizeof(T)) || !aligned(ret, sizeof(T)))
        return fail(FG_ERR_ARG, "%s: reward / value / final_value / adv / ret must be aligned to the real type", who);
    // grid-stride over columns with one wave of resident CTAs: SM count x CTAs per SM at the kernel's register count
    int dev = 0, sms = 0, per_sm = 0;
    cudaError_t err = cudaGetDevice(&dev);
    if (err == cudaSuccess) err = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (err == cudaSuccess) err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_gae<T>, kThreads, 0);
    if (err != cudaSuccess) {
        snprintf(fgabi::g_err, sizeof(fgabi::g_err), "%s: %s", who, cudaGetErrorString(err));
        return FG_ERR_CUDA;
    }
    const long long M = E * N, cap = (long long)sms * (per_sm > 0 ? per_sm : 1);
    long long blocks = (M + kThreads - 1) / kThreads;
    if (blocks > cap) blocks = cap;
    k_gae<T><<<(unsigned)blocks, kThreads, 0, (cudaStream_t)stream>>>(
        (const T*)reward, (const T*)value, (const T*)final_value, done, (T*)adv, (T*)ret, T_, E, N, (T)gamma,
        (T)(gamma * lambda));
    return launch_status(who);
}

}  // namespace

extern "C" {

int fg_gae(const void* reward, const void* value, const void* final_value, const uint8_t* done, void* adv, void* ret,
           int T, long long E, int N, double gamma, double lambda, void* stream) {
    return gae_impl<float>(reward, value, final_value, done, adv, ret, T, E, N, gamma, lambda, stream, "fg_gae");
}

int fg_gae_f64(const void* reward, const void* value, const void* final_value, const uint8_t* done, void* adv,
               void* ret, int T, long long E, int N, double gamma, double lambda, void* stream) {
    return gae_impl<double>(reward, value, final_value, done, adv, ret, T, E, N, gamma, lambda, stream, "fg_gae_f64");
}

}  // extern "C"
