// fg_lm.cuh -- host side of the warp-autonomous kernel for the partial-observation scenarios (fg_warp_lm.cuh):
// the table of instantiations.  Included by fg_lm_f32.cu / fg_lm_f64.cu only, so that these
// kernels compile in parallel with the other translation units.
#pragma once
#include "fg_abi_impl.cuh"
#include "fg_warp_lm.cuh"

namespace {

template <typename T, int N, int L, int SCN, int NOBS, bool EXT>
int launch_lm_ext(const fg::KArgs<T>& a, cudaStream_t st) {
    constexpr bool STD = std::is_same<T, float>::value;            // fp32: the standard configuration only (caller checked)
    return launch_persistent<fg::k_lm_warp<T, N, L, SCN, NOBS, STD, EXT>, fg::LmLayout<T, N, L, SCN, NOBS>>(a, "k_lm_warp", st);
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
    // the fp32 kernels are compiled for the standard product configuration only (fg_warp_lm.cuh, STD)
    if (std::is_same<T, float>::value && !std_config(a)) return 1;
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
