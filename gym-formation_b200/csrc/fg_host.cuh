#pragma once
// fg_host.cuh -- host plumbing shared by the translation units of the C ABI: the fg_last_error text, the A/B switches,
// NVTX ranges and the checks around a launch.  Definitions of g_err and switches() live in fg_abi_f32.cu.
#include <cuda_runtime.h>
#include <atomic>
#include <cstdio>
#include <nvtx3/nvToolsExt.h>

#include "../../include/formation_gym_b200.h"

namespace fgabi {
extern thread_local char g_err[512];                          // shared by every translation unit

// A/B switches for tests and profiling (fg_set_option / FG_<NAME> environment variables, read ONCE when the
// library is first used -- never on the launch path).  Defaults select the product kernels.
struct Switches {
    std::atomic<int> no_fast_pairs{0};      // tile kernel: scalar pair loops instead of fg_pairs.cuh
    std::atomic<int> force_fast_pairs{0};   // tile kernel: packed pair loops also for 32 <= N < 64 with observations
    std::atomic<int> no_cells{0};           // packed pair loops: O(N^2) group filters instead of the cell lists
    std::atomic<int> row_nbuf{2};           // OM == 2: staging buffers per warp (1 or 2)
    std::atomic<int> no_early_rows{0};      // OM == 2: rows leave after the reward pass
    std::atomic<int> no_tile_image{0};      // OM == 3 off: flat item loop
    std::atomic<int> force_tile_kernel{0};  // fg_step_fused never takes the warp-autonomous kernel
    std::atomic<int> waves{1};              // warp kernel: grid = waves x one resident wave (>= 1)
    std::atomic<int> no_std_kernel{0};      // warp kernel: never the STD instantiation (standard configuration, flags compiled out)
    std::atomic<int> l2_prefetch{1};        // warp kernel: prefetch.global.L2 of the state two spans ahead: 0 never, 1 auto, 2 always
    std::atomic<int> pf_spans{2};           // ... how many spans ahead (2 .. 8)
    std::atomic<int> row_chunks{1};         // OM == 2: chunked row writer (RC whole rows per image, one bulk store per chunk)
    std::atomic<int> row_chunk_max_log2{7}; // chunked row writer: at most 2^k rows per chunk
    std::atomic<int> row_min_n{10};         // OM == 2 (bulk-store row writers) from this agent count up
    std::atomic<int> nvtx{1};               // NVTX ranges around the launches of every entry point
};
Switches& switches();
}  // namespace fgabi

namespace {

using fgabi::g_err;

int fail(int code, const char* fmt, const char* detail = "") {
    snprintf(g_err, sizeof(g_err), fmt, detail);
    return code;
}

// After the launches of a call: FG_OK, or FG_ERR_CUDA with the launch error, prefixed by the entry point when given.
int launch_status(const char* who = "") {
    const cudaError_t err = cudaGetLastError();
    if (err == cudaSuccess) return FG_OK;
    snprintf(g_err, sizeof(g_err), "%s%skernel launch failed: %s", who, *who ? ": " : "", cudaGetErrorString(err));
    return FG_ERR_CUDA;
}

// NVTX range around the launches of one entry point (free when no tool is attached: one load + branch)
struct NvtxRange {
    bool on;
    explicit NvtxRange(const char* name) : on(fgabi::switches().nvtx.load(std::memory_order_relaxed) != 0) {
        if (on) nvtxRangePushA(name);
    }
    ~NvtxRange() { if (on) nvtxRangePop(); }
};

// cudaFuncAttributeMaxDynamicSharedMemorySize is sticky per (function, device): raise it only when a launch needs
// more than what was set before (it used to be re-set on every launch: ~1 us of host time per step).
constexpr int kMaxDev = 64;
template <auto Kernel>
cudaError_t ensure_dyn_smem(size_t smem) {
    static std::atomic<size_t> have[kMaxDev];
    if (smem <= 48 * 1024) return cudaSuccess;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDev)
        return cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (smem <= have[dev].load(std::memory_order_acquire)) return cudaSuccess;
    cudaError_t e = cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) have[dev].store(smem, std::memory_order_release);
    return e;
}

}  // namespace
