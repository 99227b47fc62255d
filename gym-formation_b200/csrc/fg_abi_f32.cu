// fg_abi_f32.cu -- fp32 entry points + the precision-independent ones (see fg_abi_impl.cuh).
#include "fg_abi_impl.cuh"
#include <cctype>

namespace fgabi {
thread_local char g_err[512] = "";

namespace {
struct OptionDesc { const char* name; std::atomic<int> Switches::* field; int lo, hi; };
const OptionDesc kOptions[] = {
    {"no_fast_pairs", &Switches::no_fast_pairs, 0, 1},       {"force_fast_pairs", &Switches::force_fast_pairs, 0, 1},
    {"no_cells", &Switches::no_cells, 0, 1},                 {"row_nbuf", &Switches::row_nbuf, 1, 2},
    {"no_early_rows", &Switches::no_early_rows, 0, 1},       {"no_tile_image", &Switches::no_tile_image, 0, 1},
    {"force_tile_kernel", &Switches::force_tile_kernel, 0, 1}, {"waves", &Switches::waves, 1, 64},
    {"nvtx", &Switches::nvtx, 0, 1},
    {"no_std_kernel", &Switches::no_std_kernel, 0, 1}, {"l2_prefetch", &Switches::l2_prefetch, 0, 2},
    {"row_chunks", &Switches::row_chunks, 0, 2}, {"row_min_n", &Switches::row_min_n, 3, 256},
    {"row_chunk_max_log2", &Switches::row_chunk_max_log2, 1, 7}, {"pf_spans", &Switches::pf_spans, 2, 8},
};
}  // namespace

// Initialised ONCE (thread-safe static) from FG_<NAME> environment variables; out-of-range values are ignored.
Switches& switches() {
    static Switches sw;
    static const bool init = [] {
        for (const OptionDesc& o : kOptions) {
            char env[64] = "FG_";
            size_t k = 3;
            for (const char* c = o.name; *c && k + 1 < sizeof(env); ++c) env[k++] = (char)toupper((unsigned char)*c);
            env[k] = 0;
            const char* v = getenv(env);
            if (!v || !*v) continue;
            char* end = nullptr;
            const long x = strtol(v, &end, 10);
            if (end != v && x >= o.lo && x <= o.hi) (sw.*(o.field)).store((int)x);
        }
        return true;
    }();
    (void)init;
    return sw;
}
}  // namespace fgabi

extern "C" {

int fg_policy_bfs(const void* pos, const void* ideal_shape, const void* ideal_vel, void* act, int E, int N,
                  int num_agents_per_layer, void* stream) {
    return policy_bfs_impl<float>(pos, ideal_shape, ideal_vel, act, E, N, num_agents_per_layer, stream);
}

int fg_abi_version(void) { return FG_ABI_VERSION; }

int fg_set_option(const char* name, int value) {
    if (!name) return fail(FG_ERR_ARG, "fg_set_option: null name%s");
    for (const fgabi::OptionDesc& o : fgabi::kOptions)
        if (!strcmp(name, o.name)) {
            if (value < o.lo || value > o.hi) return fail(FG_ERR_ARG, "fg_set_option: value out of range for '%s'", name);
            (fgabi::switches().*(o.field)).store(value);
            return FG_OK;
        }
    return fail(FG_ERR_ARG, "fg_set_option: unknown option '%s'", name);
}

int fg_get_option(const char* name, int* value) {
    if (!name || !value) return fail(FG_ERR_ARG, "fg_get_option: null argument%s");
    for (const fgabi::OptionDesc& o : fgabi::kOptions)
        if (!strcmp(name, o.name)) { *value = (fgabi::switches().*(o.field)).load(); return FG_OK; }
    return fail(FG_ERR_ARG, "fg_get_option: unknown option '%s'", name);
}

const char* fg_last_error(void) { return g_err; }

int fg_device_info(int* sm_count, int* cc_major, int* cc_minor) {
    int dev = 0;
    cudaError_t err = cudaGetDevice(&dev);
    cudaDeviceProp prop;
    if (err == cudaSuccess) err = cudaGetDeviceProperties(&prop, dev);
    if (err != cudaSuccess) return fail(FG_ERR_CUDA, "fg_device_info: %s", cudaGetErrorString(err));
    if (sm_count) *sm_count = prop.multiProcessorCount;
    if (cc_major) *cc_major = prop.major;
    if (cc_minor) *cc_minor = prop.minor;
    return FG_OK;
}

int fg_launch_geometry(int N, int* envs_per_cta, int* threads_per_cta) {
    if (N < 1 || N > FG_MAX_AGENTS) return fail(FG_ERR_ARG, "N must be in [1, FG_MAX_AGENTS=256]%s");
    if (envs_per_cta) *envs_per_cta = fg::kBlock / N;
    if (threads_per_cta) *threads_per_cta = fg::kBlock;
    return FG_OK;
}

int fg_pair_distances(const void* ent_pos, const void* ent_size, int E, int M, void* dist_vect, void* dist_mag,
                      uint8_t* collisions, void* min_dists, void* stream) {
    return pair_distances_impl<float>(ent_pos, ent_size, E, M, dist_vect, dist_mag, collisions, min_dists, stream);
}

int fg_world_step(const fg_params* p, const fg_buffers* b, int E, int N, uint64_t seed, uint32_t tick,
                  uint32_t env_offset, void* stream) {
    return world_step_impl<float>(p, b, E, N, seed, tick, env_offset, stream);
}

int fg_obs_reward(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L, void* stream) {
    return obs_reward_impl<float>(p, b, scenario, E, N, L, stream);
}

int fg_step_fused(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L, int n_steps,
                  int random_actions, int auto_reset, uint64_t seed, uint32_t tick, uint32_t env_offset,
                  void* stream) {
    return step_fused_impl<float>(p, b, scenario, E, N, L, n_steps, random_actions, auto_reset, seed, tick,
                                  env_offset, stream, nullptr, nullptr);
}

int fg_step_fused_targets(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L, int n_steps,
                          int random_actions, int auto_reset, uint64_t seed, uint32_t tick, uint32_t env_offset,
                          void* stream, const fg_targets* t) {
    return step_fused_impl<float>(p, b, scenario, E, N, L, n_steps, random_actions, auto_reset, seed, tick,
                                  env_offset, stream, t, nullptr);
}

int fg_step_fused_final(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L, int n_steps,
                        int random_actions, int auto_reset, uint64_t seed, uint32_t tick, uint32_t env_offset,
                        void* stream, const fg_targets* t, const fg_final* f) {
    return step_fused_impl<float>(p, b, scenario, E, N, L, n_steps, random_actions, auto_reset, seed, tick,
                                  env_offset, stream, t, f);
}

int fg_final_obs(const fg_params* p, const fg_final* f, const uint8_t* done, void* obs, int scenario, int E,
                 int N, int L, void* stream) {
    return final_obs_impl<float>(p, f, done, obs, scenario, E, N, L, stream);
}

int fg_obs_gather(const fg_params* p, const fg_final* states, long long R, const int64_t* rows, int B, void* obs,
                  int scenario, int N, int L, void* stream) {
    return obs_gather_impl<float>(p, states, R, rows, B, obs, scenario, N, L, stream);
}

int fg_reset(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L, const uint8_t* mask,
             uint64_t seed, uint32_t tick, uint32_t env_offset, void* stream) {
    return reset_impl<float>(p, b, scenario, E, N, L, mask, seed, tick, env_offset, stream, nullptr);
}

int fg_reset_targets(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L, const uint8_t* mask,
                     uint64_t seed, uint32_t tick, uint32_t env_offset, void* stream, const fg_targets* t) {
    return reset_impl<float>(p, b, scenario, E, N, L, mask, seed, tick, env_offset, stream, t);
}

int fg_random_actions(void* act, int E, int N, uint64_t seed, uint32_t tick, uint32_t env_offset,
                      const uint32_t* tick_dev, void* stream) {
    return random_actions_impl<float>(act, E, N, seed, tick, env_offset, tick_dev, stream);
}

}  // extern "C"
