// fg_abi_f64.cu -- fp64 entry points (the 1e-9 parity build; see fg_abi_impl.cuh).
#include "fg_abi_impl.cuh"

extern "C" {

int fg_policy_bfs_f64(const void* pos, const void* ideal_shape, const void* ideal_vel, void* act, int E, int N,
                      int num_agents_per_layer, void* stream) {
    return policy_bfs_impl<double>(pos, ideal_shape, ideal_vel, act, E, N, num_agents_per_layer, stream);
}

int fg_pair_distances_f64(const void* ent_pos, const void* ent_size, int E, int M, void* dist_vect, void* dist_mag,
                      uint8_t* collisions, void* min_dists, void* stream) {
    return pair_distances_impl<double>(ent_pos, ent_size, E, M, dist_vect, dist_mag, collisions, min_dists, stream);
}

int fg_world_step_f64(const fg_params* p, const fg_buffers* b, int E, int N, uint64_t seed, uint32_t tick,
                      uint32_t env_offset, void* stream) {
    return world_step_impl<double>(p, b, E, N, seed, tick, env_offset, stream);
}

int fg_obs_reward_f64(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L, void* stream) {
    return obs_reward_impl<double>(p, b, scenario, E, N, L, stream);
}

int fg_step_fused_f64(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L, int n_steps,
                      int random_actions, int auto_reset, uint64_t seed, uint32_t tick, uint32_t env_offset,
                      void* stream) {
    return step_fused_impl<double>(p, b, scenario, E, N, L, n_steps, random_actions, auto_reset, seed, tick,
                                   env_offset, stream, nullptr, nullptr);
}

int fg_step_fused_targets_f64(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L, int n_steps,
                              int random_actions, int auto_reset, uint64_t seed, uint32_t tick, uint32_t env_offset,
                              void* stream, const fg_targets* t) {
    return step_fused_impl<double>(p, b, scenario, E, N, L, n_steps, random_actions, auto_reset, seed, tick,
                                   env_offset, stream, t, nullptr);
}

int fg_step_fused_final_f64(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L, int n_steps,
                            int random_actions, int auto_reset, uint64_t seed, uint32_t tick, uint32_t env_offset,
                            void* stream, const fg_targets* t, const fg_final* f) {
    return step_fused_impl<double>(p, b, scenario, E, N, L, n_steps, random_actions, auto_reset, seed, tick,
                                   env_offset, stream, t, f);
}

int fg_final_obs_f64(const fg_params* p, const fg_final* f, const uint8_t* done, void* obs, int scenario, int E,
                     int N, int L, void* stream) {
    return final_obs_impl<double>(p, f, done, obs, scenario, E, N, L, stream);
}

int fg_obs_gather_f64(const fg_params* p, const fg_final* states, long long R, const int64_t* rows, int B, void* obs,
                      int scenario, int N, int L, void* stream) {
    return obs_gather_impl<double>(p, states, R, rows, B, obs, scenario, N, L, stream);
}

int fg_reset_f64(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L, const uint8_t* mask,
                 uint64_t seed, uint32_t tick, uint32_t env_offset, void* stream) {
    return reset_impl<double>(p, b, scenario, E, N, L, mask, seed, tick, env_offset, stream, nullptr);
}

int fg_reset_targets_f64(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L, const uint8_t* mask,
                         uint64_t seed, uint32_t tick, uint32_t env_offset, void* stream, const fg_targets* t) {
    return reset_impl<double>(p, b, scenario, E, N, L, mask, seed, tick, env_offset, stream, t);
}

int fg_random_actions_f64(void* act, int E, int N, uint64_t seed, uint32_t tick, uint32_t env_offset,
                          const uint32_t* tick_dev, void* stream) {
    return random_actions_impl<double>(act, E, N, seed, tick, env_offset, tick_dev, stream);
}

}  // extern "C"
