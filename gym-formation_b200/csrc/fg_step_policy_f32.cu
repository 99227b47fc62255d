// fg_step_policy_f32.cu -- fp32 entry points of the step + device controller call (fg_step_policy.cuh).  Its own
// translation unit: the POL instantiations of the warp kernel compile in parallel with the other entry points.
#include "fg_step_policy.cuh"

extern "C" int fg_step_policy(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L, int n_steps,
                              int num_agents_per_layer, int auto_reset, uint64_t seed, uint32_t tick,
                              uint32_t env_offset, void* stream) {
    return step_policy_impl<float>(p, b, scenario, E, N, L, n_steps, num_agents_per_layer, auto_reset, seed, tick,
                                   env_offset, stream, nullptr, nullptr, &fg_step_fused_final, &fg_policy_bfs);
}

extern "C" int fg_step_policy_targets(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L,
                                      int n_steps, int num_agents_per_layer, int auto_reset, uint64_t seed,
                                      uint32_t tick, uint32_t env_offset, void* stream, const fg_targets* t) {
    return step_policy_impl<float>(p, b, scenario, E, N, L, n_steps, num_agents_per_layer, auto_reset, seed, tick,
                                   env_offset, stream, t, nullptr, &fg_step_fused_final, &fg_policy_bfs);
}

extern "C" int fg_step_policy_final(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L,
                                    int n_steps, int num_agents_per_layer, int auto_reset, uint64_t seed,
                                    uint32_t tick, uint32_t env_offset, void* stream, const fg_targets* t,
                                    const fg_final* f) {
    return step_policy_impl<float>(p, b, scenario, E, N, L, n_steps, num_agents_per_layer, auto_reset, seed, tick,
                                   env_offset, stream, t, f, &fg_step_fused_final, &fg_policy_bfs);
}
