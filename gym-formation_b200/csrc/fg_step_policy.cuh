// fg_step_policy.cuh -- fg_step_policy[_f64]: env step + the reference's demo controller in one call (sm_100a).
//
// The reference's demo loop (test.py:14-28 without -r) is, per step,
//     act_n = get_action_BFS(ezpolicy, obs_n, n);  obs_n, reward_n, done_n, _ = env.step(act_n)
// Here the state stays on the device, so the loop body is "step on the action buffer, then refill the action buffer
// from the new state".  Where an instantiation exists -- formation_hd_env on the warp-autonomous kernel with
// N = n^k agents, (N, n) in {(3,3), (4,2), (8,2), (16,4)} -- that is ONE launch: the controller runs at the end
// of k_hd_warp<.., POL = n> on the positions / ideal shape / ideal_vel the step already holds on chip (fg_warp.cuh).
// Everything else (other N = n^k, tracked landmarks, per-agent constants, walls, ...) runs the same two kernels a
// caller would launch: fg_step_fused then fg_policy_bfs, n_steps times.
//
// Which shapes are fused is a measurement (B200, us per step, controller kernel + step kernel -> one fused kernel;
// scripts/policy_fused_time.py): N=3 x 1 M envs 117.3 -> 101.3, N=4 x 512 K 80.9 -> 73.2, N=8 x 128 K 58.7 -> 55.9,
// N=16 x 64 K 93.1 -> 88.6; at 4096 envs of 3 agents 7.2 -> 5.8.  Deeper / wider trees LOSE and are not dispatched
// here: N=9 x 128 K 71.7 -> 80.4, N=27 x 64 K 252.4 -> 274.5, N=25 x 64 K 284.4 -> 303.6.  In the warp layout every lane evaluates the nodes of its own
// leaders, so an upper layer costs a full warp-instruction stream for N/nxt useful lanes per env, where k_policy_bfs
// compacts the leaders of 28 envs onto consecutive threads (3 c0 + 8 c1 warp streams per 28 envs against c0 + c1 per 3),
// and the step kernel at N = 9 is already within a few per cent of being issue-bound.
#pragma once
#include "fg_abi_impl.cuh"

namespace {

template <typename T, int N, int POL>
int launch_warp_pol(const fg::KArgs<T>& a, cudaStream_t st) {
    // fp32: the standard product configuration only (STD instantiation; std_config); fp64: the generic one
    constexpr bool STD = std::is_same<T, float>::value;
    return a.obs ? launch_warp_n<T, N, true, fg::kScnHD, STD, POL>(a, st)
                 : launch_warp_n<T, N, false, fg::kScnHD, STD, POL>(a, st);
}

template <typename T>
int step_policy_impl(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L, int n_steps,
                     int n, int auto_reset, uint64_t seed, uint32_t tick, uint32_t env_offset, void* stream,
                     const fg_targets* tg, const fg_final* fin,
                     int (*step_fused)(const fg_params*, const fg_buffers*, int, int, int, int, int, int, int, uint64_t,
                                       uint32_t, uint32_t, void*, const fg_targets*, const fg_final*),
                     int (*policy_bfs)(const void*, const void*, const void*, void*, int, int, int, void*)) {
    NvtxRange nvtx_("fg_step_policy");
    int rc = check_targets<T>(tg, scenario, "fg_step_policy_targets");
    if (rc) return rc;
    rc = check_final<T>(fin, p, scenario, auto_reset, n_steps, true, "fg_step_policy_final");
    if (rc) return rc;
    if (scenario != FG_SCENARIO_HD)
        return fail(FG_ERR_ARG, "fg_step_policy: the controller reads formation_hd_env observations "
                                "(ideal_shape / ideal_vel; formation_gym/__init__.py:19-47)%s");
    if (n_steps < 1) return fail(FG_ERR_ARG, "fg_step_policy: n_steps must be >= 1%s");
    if (n < 2 || n > fg::kPolicyMaxFan) return fail(FG_ERR_ARG, "fg_step_policy: num_agents_per_layer must be in [2, 8]%s");
    const PolicyTree tree = policy_tree(N, n);
    if (!tree.levels)
        return fail(FG_ERR_ARG, "fg_step_policy: N must be a power of num_agents_per_layer ('Observation shape error!')%s");
    if (!p || !b) return fail(FG_ERR_ARG, "null params/buffers%s");
    if (!b->act || !b->pos || !b->ideal_shape || !b->ideal_vel)
        return fail(FG_ERR_ARG, "fg_step_policy: act/pos/ideal_shape/ideal_vel must be non-null%s");
    if (!p->silent) return fail(FG_ERR_ARG, "fg_step_policy: silent agents only (the controller emits no comm action)%s");

    fg::KArgs<T> a;
    rc = fill_args<T>(a, p, b, scenario, E, N, L, seed, tick, env_offset);
    if (rc) return rc;
    set_targets<T>(a, tg);
    set_final<T>(a, fin, p, scenario);
    // (fp64 has no STD instantiation: every configuration the warp path takes is fused)
    const bool fused = b->vel && b->reward && b->done && b->step && warp_path_ok<T>(a, scenario, p, b) &&
                       (!std::is_same<T, float>::value || std_config<T>(a));
    if (fused) {
        a.random_actions = 0; a.auto_reset = auto_reset;
        for (int l = 0; l < tree.levels; ++l) a.pol_mult[l] = (T)tree.mult[l];
        cudaStream_t st = (cudaStream_t)stream;
        // fp32 runs the STD instantiation, which is compiled for one step per launch: a rollout is n_steps launches
        // (with a device tick the kernel advances it itself; otherwise the tick argument counts the steps)
        const int launches = std::is_same<T, float>::value ? n_steps : 1;
        a.n_steps = std::is_same<T, float>::value ? 1 : n_steps;
        for (int ts = 0; ts < launches; ++ts) {
            a.tick = tick + (b->tick_dev ? 0u : (uint32_t)ts);
            switch (N * 16 + n) {
                case 3 * 16 + 3: rc = launch_warp_pol<T, 3, 3>(a, st); break;
                case 4 * 16 + 2: rc = launch_warp_pol<T, 4, 2>(a, st); break;
                case 8 * 16 + 2: rc = launch_warp_pol<T, 8, 2>(a, st); break;
                case 16 * 16 + 4: rc = launch_warp_pol<T, 16, 4>(a, st); break;
                default: rc = 1; break;                             // (> 0: no instantiation for this tree shape)
            }
            if (rc == 1) break;
            if (rc) return rc;
        }
        if (rc == FG_OK) return FG_OK;
    }
    // two launches per step: the kernels a caller would launch itself (same results as the fused form)
    for (int ts = 0; ts < n_steps; ++ts) {
        rc = step_fused(p, b, scenario, E, N, L, 1, 0, auto_reset, seed, tick + (b->tick_dev ? 0u : (uint32_t)ts),
                        env_offset, stream, tg, fin);
        if (rc) return rc;
        rc = policy_bfs(b->pos, b->ideal_shape, b->ideal_vel, const_cast<void*>(b->act), E, N, n, stream);
        if (rc) return rc;
    }
    return FG_OK;
}

}  // namespace
