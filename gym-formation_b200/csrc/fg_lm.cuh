// fg_lm.cuh -- host side of the warp-autonomous kernel for the partial-observation scenarios (fg_warp_lm.cuh):
// launch geometry and the table of instantiations.  Included by fg_lm_f32.cu / fg_lm_f64.cu only, so that these
// kernels compile in parallel with the other translation units.
#pragma once
#include "fg_abi_impl.cuh"
#include "fg_warp_lm.cuh"

namespace {

template <typename T, int N, int L, int SCN, int NOBS, bool STD, bool EXT>
const WarpGeom& lm_geom() {
    static const WarpGeom geom = [] {
        typedef fg::LmLayout<T, N, L, SCN, NOBS> LY;
        WarpGeom g_; g_.best = 0; g_.sms = 148;
        int dev = 0;
        if (cudaGetDevice(&dev) == cudaSuccess)
            cudaDeviceGetAttribute(&g_.sms, cudaDevAttrMultiProcessorCount, dev);
        int best_res = -1;
        for (int l = 3; l >= 0; --l) {
            const int w = 1 << l;
            const size_t smem = (size_t)w * LY::stride;
            g_.ctas[l] = 0;
            if (smem > 227 * 1024 || w > LY::MAXW) continue;
            if (cudaFuncSetAttribute(fg::k_lm_warp<T, N, L, SCN, NOBS, STD, EXT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)smem) != cudaSuccess) { cudaGetLastError(); continue; }
            int ctas = 0;
            if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas, fg::k_lm_warp<T, N, L, SCN, NOBS, STD, EXT>, 32 * w, smem)
                != cudaSuccess) { cudaGetLastError(); continue; }
            g_.ctas[l] = ctas;
            if (ctas * w > best_res) { best_res = ctas * w; g_.best = l; }
        }
        // (see warp_geom: the probing left the limit at the smallest footprint)
        cudaFuncSetAttribute(fg::k_lm_warp<T, N, L, SCN, NOBS, STD, EXT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 48 * 1024);
        cudaGetLastError();
        return g_;
    }();
    return geom;
}

template <typename T, int N, int L, int SCN, int NOBS, bool EXT>
int launch_lm_ext(const fg::KArgs<T>& a, cudaStream_t st) {
    constexpr bool STD = std::is_same<T, float>::value;            // fp32: the standard configuration only (caller checked)
    typedef fg::LmLayout<T, N, L, SCN, NOBS> LY;
    const WarpGeom& gm = lm_geom<T, N, L, SCN, NOBS, STD, EXT>();
    const int spans = (a.E + LY::EPW - 1) / LY::EPW;
    int l = gm.best;
    while (l > 0 && (spans >> l) < 2 * gm.sms) --l;                // small batches: spread over the SMs
    if (gm.ctas[l] < 1) return fail(FG_ERR_CUDA, "k_lm_warp does not fit on this device%s");
    const int w = 1 << l;
    const size_t smem = (size_t)w * LY::stride;
    cudaError_t err = ensure_dyn_smem<fg::k_lm_warp<T, N, L, SCN, NOBS, STD, EXT>>(smem);
    if (err != cudaSuccess) return fail(FG_ERR_CUDA, "cudaFuncSetAttribute failed: %s", cudaGetErrorString(err));
    int grid = (spans + w - 1) / w;                                // persistent warps: at most one resident wave
    int wave = gm.sms * gm.ctas[l];
    wave *= std::max(1, fgabi::switches().waves.load(std::memory_order_relaxed));
    if (grid > wave) grid = wave;
    if ((grid * w) & 1) ++grid;                                    // even warp count (16-byte phase, fg_warp.cuh)
    fg::k_lm_warp<T, N, L, SCN, NOBS, STD, EXT><<<grid, 32 * w, smem, st>>>(a);
    err = cudaGetLastError();
    if (err != cudaSuccess) return fail(FG_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(err));
    return FG_OK;
}

// runs with a terminal block take the EXT instantiation of the same kernel
template <typename T, int N, int L, int SCN, int NOBS>
int launch_lm_n(const fg::KArgs<T>& a, cudaStream_t st) {
    if (fg::reset_ext(a)) return launch_lm_ext<T, N, L, SCN, NOBS, true>(a, st);
    return launch_lm_ext<T, N, L, SCN, NOBS, false>(a, st);
}

// Instantiations: make_world's default landmark counts (5 / 4) and num_obs = 3 for 3 .. 9 agents -- what
// make_env(scenario, num_agents = n) builds (formation_gym/__init__.py:6-17).  Returns 1 when there is none.
template <typename T>
int launch_lm_dispatch(const fg::KArgs<T>& a, int scenario, cudaStream_t st) {
    if (std::is_same<T, float>::value) {
        // the fp32 kernels are compiled for the standard product configuration (fg_warp_lm.cuh, STD)
        const bool std_cfg = a.collide && !a.has_vmax && a.mass_one && a.n_steps == 1 &&
                             a.step && a.done && a.indiv && a.ep_return && a.ep_coll && a.stats && !a.comm &&
                             !fgabi::switches().no_std_kernel.load(std::memory_order_relaxed);
        if (!std_cfg) return 1;
    }
    if (scenario == FG_SCENARIO_HD_PARTIAL && a.L == 5 && a.num_obs == 3) {
        switch (a.N) {
            case 3: return launch_lm_n<T, 3, 5, fg::kScnPartial, 3>(a, st);
            case 4: return launch_lm_n<T, 4, 5, fg::kScnPartial, 3>(a, st);
            case 5: return launch_lm_n<T, 5, 5, fg::kScnPartial, 3>(a, st);
            case 6: return launch_lm_n<T, 6, 5, fg::kScnPartial, 3>(a, st);
            case 7: return launch_lm_n<T, 7, 5, fg::kScnPartial, 3>(a, st);
            case 8: return launch_lm_n<T, 8, 5, fg::kScnPartial, 3>(a, st);
            case 9: return launch_lm_n<T, 9, 5, fg::kScnPartial, 3>(a, st);
            default: return 1;
        }
    }
    if (scenario == FG_SCENARIO_HD_PARTIAL_RANGE && a.L == 4) {
        switch (a.N) {
            case 3: return launch_lm_n<T, 3, 4, fg::kScnRange, 0>(a, st);
            case 4: return launch_lm_n<T, 4, 4, fg::kScnRange, 0>(a, st);
            case 5: return launch_lm_n<T, 5, 4, fg::kScnRange, 0>(a, st);
            case 6: return launch_lm_n<T, 6, 4, fg::kScnRange, 0>(a, st);
            case 7: return launch_lm_n<T, 7, 4, fg::kScnRange, 0>(a, st);
            case 8: return launch_lm_n<T, 8, 4, fg::kScnRange, 0>(a, st);
            case 9: return launch_lm_n<T, 9, 4, fg::kScnRange, 0>(a, st);
            default: return 1;
        }
    }
    // formation_hd_obs_env: make_world's 4 goal landmarks + 3 obstacles (formation_hd_obs_env.py:14)
    if (scenario == FG_SCENARIO_HD_OBSTACLE && a.L == 7 && a.n_obst == 3 && a.n_walls == 0) {
        switch (a.N) {
            case 3: return launch_lm_n<T, 3, 7, fg::kScnObstacle, 3>(a, st);
            case 4: return launch_lm_n<T, 4, 7, fg::kScnObstacle, 3>(a, st);
            case 5: return launch_lm_n<T, 5, 7, fg::kScnObstacle, 3>(a, st);
            case 6: return launch_lm_n<T, 6, 7, fg::kScnObstacle, 3>(a, st);
            case 7: return launch_lm_n<T, 7, 7, fg::kScnObstacle, 3>(a, st);
            case 8: return launch_lm_n<T, 8, 7, fg::kScnObstacle, 3>(a, st);
            case 9: return launch_lm_n<T, 9, 7, fg::kScnObstacle, 3>(a, st);
            default: return 1;
        }
    }
    return 1;
}

}  // namespace
