// fg_warp_lm.cuh -- warp-autonomous fused step kernel for the partial-observation scenarios (sm_100a):
// formation_hd_partial_env (formation_gym/envs/formation_hd_partial_env.py:15-125) and
// formation_hd_partial_range_env (formation_hd_partial_range_env.py:15-113) at the agent counts the reference's own
// training recipes use (train/README.md:40,51,173: 4 and 5 agents; here N = 3 .. 9).
//
// Why it exists: these scenarios ran on the generic tile kernel, which at N = 4 / 5 is issue-bound (per-item index
// arithmetic and six CTA barriers per step): 0.37-0.44 of the HBM peak (262144 envs; DESIGN.md section 3.1b) where the
// formation_hd_env kernel of the same layout reaches 0.79-0.91.  This is that kernel's design (fg_warp.cuh: lane <->
// agent, EPW = floor(32 / N) whole envs per warp, __syncwarp() only, persistent warps with a register prefetch of the
// next span, the span's observation rows leaving the SM as ONE TMA bulk store) for worlds whose landmarks are
// free-standing entities:
//   * L landmarks per env, L != N in general (make_world's defaults: 5 for the partial scenario, 4 for the range
//     one, whatever num_agents is -- formation_gym/__init__.py:11 passes only num_agents).  A span's landmarks are
//     EPW * L consecutive items of lm[E,L,2]; lane q copies items q, q + 32, ... of the NEXT span into shared memory
//     with cp.async while this span is computed.
//   * reward = -max(dH(u, v), dH(v, u)) of the agents and the landmarks, each centred on its own mean
//     (formation_hd_partial_env.py:67-75), minus one per collision; no velocity term.  Lane i owns row i (min over
//     the landmarks) and the columns of landmarks i, i + N, ... (min over the agents).
//   * row = [p_vel | landmark positions (absolute) | other_pos | comm zeros (N-1)]: other_pos are the NOBS agents after
//     me in cyclic order (partial, :50-53) or all others clipped to +-obs_range (range, :49-52).
//   * formation_hd_obs_env (formation_gym/envs/formation_hd_obs_env.py:14-149; train/README.md:43,53,171: 4 agents): the
//     last NO landmarks are movable colliding obstacles.  Lane i < NO of an env also owns obstacle i: its contact forces
//     against the agents and the other obstacles in the reference's entity order, its integration, the reward hook's
//     velocity rule and its reset (semantics: fg_obstacle.cuh, whose tile kernel stays the fallback).  The reward is the
//     goals' Hausdorff term minus 2 per collision with an agent or an obstacle; the obstacles enter the row relative to
//     the agent.
// Restrictions (host: lm_warp_ok in fg_abi_impl.cuh): uniform agent constants, no walls, silent agents, an
// observation buffer; anything else takes the tile kernel, which implements the same semantics (and is what the fp64
// goldens of the unmodified reference pin; tests compare the two kernels and each against the oracle).
#pragma once
#include "fg_kernels.cuh"
#include "fg_obstacle.cuh"

namespace fg {

template <typename T, int N, int L, int SCN, int NOBS> struct LmLayout {
    typedef typename Ops<T>::R2 R2;
    typedef typename Ops<T>::Bits Bits;
    static constexpr int EPW = 32 / N;                 // envs per warp
    static constexpr int NA = EPW * N;                 // active lanes
    static constexpr int NL = EPW * L;                 // landmarks of a span
    static constexpr int NLR = (NL + 31) / 32;         // landmark items per lane
    // formation_hd_obs_env: L = goal landmarks + obstacles (world.landmarks order), NOBS = the number of obstacles;
    // its row [p_vel | goals (LG) | obstacles - p (NO) | other_pos (N-1) | comm (N-1)] has the range scenario's length
    static constexpr int NO = (SCN == kScnObstacle) ? NOBS : 0;     // movable colliding obstacles (the last NO landmarks)
    static constexpr int LG = L - NO;                               // goal landmarks
    static constexpr int NREL = (SCN == kScnPartial) ? NOBS : N - 1;
    static constexpr int IPR = 1 + L + NREL + (N - 1); // R2 items per observation row
    static constexpr int MAXW = 8;
    static constexpr size_t off_obs = 0;                                     // +16 B slack for the 8-byte phase
    static constexpr size_t off_pold = off_obs + (size_t)NA * IPR * sizeof(R2) + 16;
    static constexpr size_t off_pnew = off_pold + (size_t)NA * sizeof(R2);   // [EPW][2N]: p_0..p_{N-1} twice
    static constexpr size_t off_cen = off_pnew + (size_t)2 * NA * sizeof(R2);
    static constexpr size_t off_vel = off_cen + (size_t)NA * sizeof(R2);
    static constexpr size_t off_lm = off_vel + (size_t)NA * sizeof(R2);      // 2 x [EPW][L] landmark positions (this span, next span)
    static constexpr size_t off_ov = off_lm + (size_t)2 * NL * sizeof(R2);   // 2 x [EPW][NO] obstacle velocities (as off_lm)
    static constexpr size_t off_on = off_ov + (size_t)2 * EPW * NO * sizeof(R2);   // [EPW][NO] obstacle positions after the step
    static constexpr size_t off_max = off_on + (size_t)EPW * NO * sizeof(R2);
    static constexpr size_t off_col = off_max + (size_t)EPW * sizeof(Bits);
    static constexpr size_t off_stat = (off_col + (size_t)EPW * sizeof(int) + 7) & ~(size_t)7;   // 4 doubles
    static constexpr size_t raw = off_stat + 4 * sizeof(double);
    static constexpr size_t stride = (raw + 15) & ~(size_t)15;
    static_assert(SCN == kScnPartial || SCN == kScnRange || SCN == kScnObstacle, "landmark scenarios");
    static_assert(NO <= N && LG >= 1, "lane i of an env also owns obstacle i");
    static_assert(N >= 2 && N <= 16 && L >= 1 && NLR <= 4, "small worlds only");
    static_assert(SCN != kScnPartial || (NOBS >= 1 && NOBS <= N), "the cyclic neighbour window fits the doubled array");
};

// STD: the standard product configuration, asserted by the host before it picks this instantiation (agents collide,
// unit mass, no max_speed, one step per launch, step / done / indiv / ep_return / ep_collisions / stats present, no comm
// buffer): the warp-uniform run-time tests of these are compiled out, as in fg_warp.cuh.  The fp32 build has only
// this instantiation (anything else takes the tile kernel), the fp64 build only the generic one.
// EXT (reset extension, as in fg_warp.cuh): the auto-reset copies the terminal state into the terminal block
// (KArgs::fin_*); its own instantiation, so that the kernels of runs without a block keep their register allocation.
template <typename T, int N, int L, int SCN, int NOBS, bool STD, bool EXT = false>
// (three 8-warp CTAs per SM, <= 80 registers: for the obstacle scenario two CTAs at up to 128 registers run 62.6 -> 69.7 us
// per 262144 envs of 4 agents, four at 64 registers with 56 bytes of spills 62.3 -> 68.4 us)
__global__ void __launch_bounds__(32 * LmLayout<T, N, L, SCN, NOBS>::MAXW, 3) k_lm_warp(const __grid_constant__ KArgs<T> a) {
    typedef Ops<T> O;
    typedef typename O::R2 R2;
    typedef typename O::Bits Bits;
    typedef LmLayout<T, N, L, SCN, NOBS> LY;
    constexpr int EPW = LY::EPW, NA = LY::NA, NL = LY::NL, NLR = LY::NLR, IPR = LY::IPR, NREL = LY::NREL;
    constexpr int NO = LY::NO, LG = LY::LG;
    constexpr bool OBST = (SCN == kScnObstacle);
    constexpr unsigned FULL = 0xffffffffu;
    extern __shared__ __align__(128) unsigned char smem_raw[];

    const bool f_collide = STD ? true : (a.collide != 0), f_noise = a.u_noise > (T)0;   // (motor noise stays a run-time flag)
    const bool f_vmax = STD ? false : (a.has_vmax != 0), f_mass1 = STD ? true : (a.mass_one != 0);
    const bool has_step = STD ? true : (a.step != nullptr), has_done = STD ? true : (a.done != nullptr);
    const bool has_indiv = STD ? true : (a.indiv != nullptr), has_epr = STD ? true : (a.ep_return != nullptr);
    const bool has_epc = STD ? true : (a.ep_coll != nullptr), has_stats = STD ? true : (a.stats != nullptr);
    const bool has_comm = STD ? false : (a.comm != nullptr);
    const int n_steps = STD ? 1 : a.n_steps;

    const int lane = threadIdx.x & 31;
    const int wib = threadIdx.x >> 5;
    const int wpc = blockDim.x >> 5;
    const int gw = blockIdx.x * wpc + wib;                                  // global warp index
    const int nwarps = gridDim.x * wpc;                                     // EVEN (host): a warp's spans keep one 16-byte phase
    const int nspans = (a.E + EPW - 1) / EPW;                               // one span = EPW consecutive envs
    if (gw >= nspans) return;                                               // warp-uniform; no CTA barriers below
    const uint32_t tick0 = a.tick + (a.tick_dev ? a.tick_dev[0] : 0u);
    const int le = lane < NA ? lane / N : 0;
    const int i = lane < NA ? lane - le * N : 0;
    const unsigned envmask = ((1u << N) - 1u) << (le * N);                  // lanes of this env

    unsigned char* wr = smem_raw + (size_t)wib * LY::stride;
    R2* s_pold = reinterpret_cast<R2*>(wr + LY::off_pold);
    R2* s_pnew = reinterpret_cast<R2*>(wr + LY::off_pnew);
    R2* s_cen = reinterpret_cast<R2*>(wr + LY::off_cen);
    R2* s_vel = reinterpret_cast<R2*>(wr + LY::off_vel);
    R2* s_lm2 = reinterpret_cast<R2*>(wr + LY::off_lm);
    R2* s_ov2 = reinterpret_cast<R2*>(wr + LY::off_ov);                     // obstacle velocities (formation_hd_obs_env)
    R2* s_on = reinterpret_cast<R2*>(wr + LY::off_on);                      // obstacle positions after the step
    Bits* s_max = reinterpret_cast<Bits*>(wr + LY::off_max);
    int* s_col = reinterpret_cast<int*>(wr + LY::off_col);
    double* s_stat = reinterpret_cast<double*>(wr + LY::off_stat);          // per-warp episode statistics (see fg_warp.cuh)
    if (lane < 4) s_stat[lane] = 0.0;

    // formation_hd_obs_env: contact geometry of the agent-obstacle and obstacle-obstacle pairs (core.py:307) and the mass
    // ratios of core.py:314-318 -- launch constants
    const T dmin_ao = OBST ? O::add(a.size, a.osize) : (T)0, dmin_oo = OBST ? O::add(a.osize, a.osize) : (T)0;
    const T cut_ao = dmin_ao + a.kcut * a.margin, cut_oo = dmin_oo + a.kcut * a.margin;
    const T cut2_ao = cut_ao * cut_ao, cut2_oo = cut_oo * cut_oo;
    const T ratio_ao = OBST ? O::div(a.omass, a.mass) : (T)1;               // force on the agent: (m_b / m_a) * force
    const T ratio_oa = OBST ? -O::div((T)1, ratio_ao) : (T)1;               // on the obstacle: -(m_a / m_b) * force
    const T dmin_ao2_hi = dmin_ao * dmin_ao * (T)1.0001;                    // guarded square: candidates of the exact test

    const R2 zero = O::make((T)0, (T)0);
    bool bulk_pending = false;
    const R2* zeroed = nullptr;                                             // image whose comm slots hold zeros

    // software pipeline over the spans of this (persistent) warp: the next span's state is in flight while this
    // one is computed -- the per-agent arrays in registers, the landmarks (up to two items per lane) through
    // cp.async straight into the other half of a double buffer: holding them in registers too made ptxas spill
    // under the 80-register bound, and with ~2 KB of L1 left beside the shared memory every spill reload is an L2
    // round trip (N = 4: long-scoreboard stalls 4.2 per issue, issue active 50 %, profiles/r02c_lm4_before_ncu_summary.json).
    R2 p_n = zero, v_n = zero, u_n = zero;
    T epr_n = (T)0;
    int stp_n = 0, epc_n = 0;
    int buf = 0;                                                            // half of s_lm2 the NEXT fetch fills
    auto fetch = [&](int span) {
        const int fe0 = span * EPW;
        const int nv = min(EPW, a.E - fe0);
        p_n = zero; v_n = zero; u_n = zero; stp_n = 0; epr_n = (T)0; epc_n = 0;
        if (lane < nv * N) {                                                // coalesced: lane <-> consecutive agent
            const size_t fa = (size_t)fe0 * N + lane;
            p_n = a.pos[fa];
            v_n = a.vel[fa];
            if (!a.random_actions) u_n = a.act[fa];
            if (has_step) stp_n = a.step[fe0 + le];
            if (i == 0) {                                                   // running episode statistics of the env
                if (has_epr) epr_n = a.ep_return[fe0 + le];
                if (has_epc) epc_n = a.ep_coll[fe0 + le];
            }
        }
#pragma unroll
        for (int r = 0; r < NLR; ++r) {
            const int q = lane + 32 * r;
            if (q < nv * L)
                asm volatile("cp.async.ca.shared.global [%0], [%1], %2;"
                             :: "r"(smem_u32(s_lm2 + buf * NL + q)), "l"(a.lm + (size_t)fe0 * L + q), "n"(sizeof(R2)) : "memory");
        }
        if (OBST && a.lmv && lane < nv * NO) {                              // landmark_vel[E,L,2]: obstacle entries only
            const int qe = lane / (NO > 0 ? NO : 1), k = lane - qe * NO;
            asm volatile("cp.async.ca.shared.global [%0], [%1], %2;"
                         :: "r"(smem_u32(s_ov2 + buf * (EPW * NO) + lane)), "l"(a.lmv + (size_t)(fe0 + qe) * L + LG + k),
                            "n"(sizeof(R2)) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        buf ^= 1;
    };
    fetch(gw);

  int spans_left = (nspans - gw + nwarps - 1) / nwarps;                     // >= 1
  for (int span = gw; ; span += nwarps) {
    const int env0 = span * EPW;
    const int nval = min(EPW, a.E - env0);
    const bool active = lane < nval * N;
    const int e = env0 + le;
    const size_t g = (size_t)env0 * N + lane;                               // global agent index
    const uint32_t ge = a.env_offset + (uint32_t)e;                         // global env id (Philox counter)
    R2* g_obs = a.obs + (size_t)env0 * N * IPR;
    const uint32_t obs_bytes = (uint32_t)(nval * N * IPR) * (uint32_t)sizeof(R2);
    const uint32_t obs_head = (uint32_t)((16u - ((uint32_t)(uintptr_t)g_obs & 15u)) & 15u);   // 0 or 8 (fp32), 0 (fp64)
    R2* s_obs = reinterpret_cast<R2*>(wr + LY::off_obs + ((16u - obs_head) & 15u));

    R2 p = p_n, v = v_n, u = u_n;
    T epr = epr_n;
    int stp = stp_n, epc = epc_n;
    R2* s_lm = s_lm2 + (buf ^ 1) * NL;                                      // filled by the fetch of the previous iteration
    R2* s_ov = s_ov2 + (buf ^ 1) * (EPW * NO);
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncwarp();                                                           // every lane's copies landed; readers of the other half are done
    if (spans_left > 1) fetch(span + nwarps);
    // formation_hd_obs_env: lane i < NO of an env also owns obstacle i (entity N + LG + i of the reference's pair loop)
    const bool obst_lane = OBST && active && i < NO;
    R2 ov = zero;                                                           // its velocity (NULL landmark_vel: at rest)
    if (obst_lane && a.lmv) ov = s_ov[le * NO + i];

    for (int ts = 0; ts < n_steps; ++ts) {
        if (lane < EPW) { s_max[lane] = 0; s_col[lane] = 0; }
        if (lane < NA) s_pold[lane] = p;
        // contact cut-offs of my env: NaN when one of its old agent or obstacle positions is not finite (env_cut2,
        // fg_kernels.cuh)
        T cut2 = a.cut2, c2_ao = cut2_ao, c2_oo = cut2_oo;
        if (f_collide || OBST) {                                            // (obstacle pairs collide whatever collide says)
            bool bad = active && nonfinite2(p.x, p.y);
            if (obst_lane) { const R2 po = s_lm[le * L + LG + i]; bad |= nonfinite2(po.x, po.y); }
            const bool env_nf = (__ballot_sync(FULL, bad) & envmask) != 0u;
            cut2 = env_cut2(a.cut2, env_nf);
            if constexpr (OBST) { c2_ao = env_cut2(cut2_ao, env_nf); c2_oo = env_cut2(cut2_oo, env_nf); }
        }
        __syncwarp();

        // =============================== World.step (core.py:206-225) ===========================
        if (active) {
            if (a.random_actions) {                                         // test.py:20
                U4 r = philox(a.seed, ge, (uint32_t)i, tick0 + (uint32_t)ts, kAction);
                u = O::make(uniform_pm1<T>(r.x), uniform_pm1<T>(r.y));
                if (a.random_actions == 2) const_cast<R2*>(a.act)[g] = u;   // recorded for the caller (replay buffer)
            }
            // _set_action: u *= sensitivity (environment.py:216-221); apply_action_force: F = gain * u + noise
            // (core.py:232-236)
            T Fx = O::mul(a.gain, O::mul(u.x, a.sens));
            T Fy = O::mul(a.gain, O::mul(u.y, a.sens));
            if (f_noise) {
                U4 r = philox(a.seed, ge, (uint32_t)i, tick0 + (uint32_t)ts, kUNoise);
                T n0, n1; normal_pair<T>(r.x, r.y, &n0, &n1);
                Fx = O::add(Fx, O::mul(n0, a.u_noise));
                Fy = O::add(Fy, O::mul(n1, a.u_noise));
            }
            // apply_environment_force (core.py:240-254): landmarks do not collide (make_world: collide = False), so
            // the pairs are agent-agent.  Near-pair bitmask first, then the softplus contact force for the set
            // bits in ascending j = the reference's accumulation order.
            if (f_collide) {
                const R2* ep = s_pold + le * N;
                unsigned near = 0;
#pragma unroll
                for (int j = 0; j < N; ++j) {
                    R2 q = ep[j];
                    T dx = O::sub(p.x, q.x), dy = O::sub(p.y, q.y);
                    T d2 = dx * dx + dy * dy;
                    near |= (!(d2 >= cut2)) ? (1u << j) : 0u;               // !(>=) keeps NaN pairs; see env_cut2
                }
                near &= ~(1u << i);
                const T dmin = O::add(a.size, a.size);                      // core.py:307
                while (near) {
                    const int j = __ffs(near) - 1;
                    near &= near - 1;
                    R2 q = ep[j];
                    T dx = (j < i) ? O::sub(q.x, p.x) : O::sub(p.x, q.x);   // delta = p_a - p_b, a < b
                    T dy = (j < i) ? O::sub(q.y, p.y) : O::sub(p.y, q.y);
                    T fx, fy;
                    contact_force<T>(dx, dy, dmin, a.margin, a.cforce, &fx, &fy);
                    if (j < i) { Fx = O::add(-fx, Fx); Fy = O::add(-fy, Fy); }   // equal masses: ratio 1
                    else       { Fx = O::add(fx, Fx);  Fy = O::add(fy, Fy); }
                }
                if constexpr (OBST) {
                    // agent (entity a) against every obstacle (entity b > a; goal landmarks do not collide,
                    // core.py:292): force_a = (m_b / m_a) * force (core.py:314-318)
                    const R2* envo = s_lm + le * L + LG;
                    const T ratio = ratio_ao;
#pragma unroll
                    for (int k = 0; k < NO; ++k) {
                        R2 q = envo[k];
                        T dx = O::sub(p.x, q.x), dy = O::sub(p.y, q.y);
                        if (!(dx * dx + dy * dy >= c2_ao)) {
                            T fx, fy;
                            contact_force<T>(dx, dy, dmin_ao, a.margin, a.cforce, &fx, &fy);
                            Fx = O::add(O::mul(ratio, fx), Fx); Fy = O::add(O::mul(ratio, fy), Fy);
                        }
                    }
                }
            }
            // integrate_state (core.py:264-277)
            v.x = O::mul(v.x, a.keep); v.y = O::mul(v.y, a.keep);
            T ax = f_mass1 ? Fx : O::div(Fx, a.mass);
            T ay = f_mass1 ? Fy : O::div(Fy, a.mass);
            v.x = O::add(v.x, O::mul(ax, a.dt));
            v.y = O::add(v.y, O::mul(ay, a.dt));
            if (f_vmax) {
                T sp = O::sqrt_(O::sq2(v.x, v.y));
                if (sp > a.vmax) {
                    v.x = O::mul(O::div(v.x, sp), a.vmax);
                    v.y = O::mul(O::div(v.y, sp), a.vmax);
                }
            }
            p.x = O::add(p.x, O::mul(v.x, a.dt));
            p.y = O::add(p.y, O::mul(v.y, a.dt));
            s_pnew[le * 2 * N + i] = p;
            s_pnew[le * 2 * N + N + i] = p;
            s_vel[lane] = v;
            if (ts == n_steps - 1) {
                a.pos[g] = p; a.vel[g] = v;
                if (has_comm) a.comm[g] = zero;                             // update_agent_state: silent -> c = 0
            }
        }
        if constexpr (OBST) {
            // the obstacles themselves (fg_obstacle.cuh): contributions in entity order -- agents (the obstacle is entity
            // b: -(m_a / m_b) * force), earlier obstacles (b), later obstacles (a); no action force, damped and
            // integrated like an agent, never speed-clamped (core.py:264-277)
            if (obst_lane) {
                const R2* envo = s_lm + le * L + LG;
                const R2 po = envo[i];
                T Fx = (T)0, Fy = (T)0;
                if (f_collide) {
                    const R2* envp = s_pold + le * N;
                    const T c = ratio_oa;
#pragma unroll
                    for (int j = 0; j < N; ++j) {
                        R2 pj = envp[j];
                        T dx = O::sub(pj.x, po.x), dy = O::sub(pj.y, po.y);
                        if (!(dx * dx + dy * dy >= c2_ao)) {
                            T fx, fy;
                            contact_force<T>(dx, dy, dmin_ao, a.margin, a.cforce, &fx, &fy);
                            Fx = O::add(O::mul(c, fx), Fx); Fy = O::add(O::mul(c, fy), Fy);
                        }
                    }
                }
#pragma unroll
                for (int m = 0; m < NO; ++m) {
                    if (m == i) continue;
                    R2 q2 = envo[m];
                    T dx = (m < i) ? O::sub(q2.x, po.x) : O::sub(po.x, q2.x);
                    T dy = (m < i) ? O::sub(q2.y, po.y) : O::sub(po.y, q2.y);
                    if (!(dx * dx + dy * dy >= c2_oo)) {
                        T fx, fy;
                        contact_force<T>(dx, dy, dmin_oo, a.margin, a.cforce, &fx, &fy);
                        if (m < i) { Fx = O::add(-fx, Fx); Fy = O::add(-fy, Fy); }     // equal obstacle masses
                        else       { Fx = O::add(fx, Fx);  Fy = O::add(fy, Fy); }
                    }
                }
                ov.x = O::mul(ov.x, a.keep); ov.y = O::mul(ov.y, a.keep);
                ov.x = O::add(ov.x, O::mul(O::div(Fx, a.omass), a.dt));
                ov.y = O::add(ov.y, O::mul(O::div(Fy, a.omass), a.dt));
                s_on[le * NO + i] = O::make(O::add(po.x, O::mul(ov.x, a.dt)), O::add(po.y, O::mul(ov.y, a.dt)));
            }
        }
        // any non-finite position in an env makes its centroid, hence the whole shape term, NaN
        const bool bad = !(fabs(p.x) < (T)INFINITY) || !(fabs(p.y) < (T)INFINITY);
        const bool env_bad = (__ballot_sync(FULL, active && bad) & envmask) != 0u;
        __syncwarp();

        // ============ Scenario.reward on the NEW state (formation_hd_partial_env.py:67-87; Q16) ============
        // u - mean(u), v - mean(v) (:70-74): np.mean sums the rows in entity order.  Every lane of an env computes both
        // means itself -- the positions from its env's lanes by shuffle, the landmarks from shared memory (every lane
        // of an env reads the same addresses: broadcasts) -- so nothing is staged and no lane waits for another.
        // (One lane per (env, mean) writing to shared memory, as fg_warp.cuh does, cost 5-way bank conflicts on the
        // strided reads and two more warp barriers: profiles/r02d_lm4_ncu_summary.json.)
        T sx = 0, sy = 0, lx = 0, ly = 0;
#pragma unroll
        for (int j = 0; j < N; ++j) {
            sx = O::add(sx, __shfl_sync(FULL, p.x, le * N + j));
            sy = O::add(sy, __shfl_sync(FULL, p.y, le * N + j));
        }
        const R2* eL = s_lm + le * L;
#pragma unroll
        for (int k = 0; k < LG; ++k) { R2 l = eL[k]; lx = O::add(lx, l.x); ly = O::add(ly, l.y); }   // (goal landmarks)
        const R2 mp = O::make(O::div_count(sx, N), O::div_count(sy, N));    // fp64: true division, as np.mean
        const R2 ml = O::make(O::div_count(lx, LG), O::div_count(ly, LG));
        const R2 C = O::make(O::sub(p.x, mp.x), O::sub(p.y, mp.y));         // centred agent shape
        if (lane < NA) s_cen[lane] = C;
        __syncwarp();

        int col = 0;
        if (active) {
            const R2* eC = s_cen + le * N;
            const R2* eP = s_pnew + le * 2 * N + i;                         // eP[k] = agent (i + k) mod N
            T dmax = (T)INFINITY;
#pragma unroll
            for (int k = 0; k < LG; ++k) {                                  // row i: min_k |C_i - V_k|^2, V_k = l_k - mean(l)
                const R2 l = eL[k];
                dmax = fmin(dmax, O::sq2(O::sub(C.x, O::sub(l.x, ml.x)), O::sub(C.y, O::sub(l.y, ml.y))));
            }
#pragma unroll
            for (int k0 = 0; k0 < LG; k0 += N) {                            // columns i, i + N, ...: min_j |C_j - V_k|^2
                const int k = k0 + i;
                if (k < LG) {
                    const R2 l = eL[k];
                    const R2 Vk = O::make(O::sub(l.x, ml.x), O::sub(l.y, ml.y));
                    T colmin = (T)INFINITY;
#pragma unroll
                    for (int j = 0; j < N; ++j) {
                        R2 Cj = eC[j];
                        colmin = fmin(colmin, O::sq2(O::sub(Cj.x, Vk.x), O::sub(Cj.y, Vk.y)));
                    }
                    dmax = fmax(dmax, colmin);
                }
            }
            // is_collision with every other agent (:82-86,123-125): exact test only for candidates
            unsigned hit = 0;
#pragma unroll
            for (int k = 1; k < N; ++k) {
                R2 q = eP[k];
                T dx = O::sub(q.x, p.x), dy = O::sub(q.y, p.y);
                T d2 = dx * dx + dy * dy;
                hit |= (d2 < a.rthr2_hi) ? (1u << k) : 0u;
            }
            while (f_collide && hit) {
                const int k = __ffs(hit) - 1;
                hit &= hit - 1;
                R2 q = eP[k];
                if (O::norm2(O::sub(q.x, p.x), O::sub(q.y, p.y)) < a.rthr) ++col;
            }
            if constexpr (OBST) {                                           // ... and with every obstacle (formation_hd_obs_env.py:91-97)
                const R2* envo = s_on + le * NO;
#pragma unroll
                for (int k = 0; k < NO; ++k) {
                    R2 q = envo[k];
                    T dx = O::sub(q.x, p.x), dy = O::sub(q.y, p.y);
                    if (f_collide && dx * dx + dy * dy < dmin_ao2_hi && O::norm2(dx, dy) < dmin_ao) ++col;
                }
            }
            atomicMax(&s_max[le], O::bits(dmax));                           // d2 >= 0: bit order == value order
            if (col) atomicAdd(&s_col[le], col);
        }
        __syncwarp();

        // ============ rewards, done, statistics (environment.py:126-138,172-177) ================
        stp += 1;                                                           // environment.py:114
        const bool dn = active && has_step && (stp >= a.world_length);
        if (active) {
            T base = -O::sqrt_(O::from_bits(s_max[le]));                    // -max(dH(u,v), dH(v,u)); no velocity term
            if (env_bad) base = O::from_bits(~(Bits)0 >> 1);                // NaN, as the reference
            constexpr int CPEN = OBST ? 2 : 1;                              // rew -= 1 (2: formation_hd_obs_env.py:93,97) per collision
            T r = base;
            for (int c = 0; c < col; ++c) r = O::sub(r, (T)CPEN);
            const int coltot = s_col[le];
            // shared reward = sum_i r_i (environment.py:136): N*base - CPEN * total collisions, in fp64
            const double R = (double)N * (double)base - (double)CPEN * (double)coltot;
            a.reward[g] = (T)R;
            if (has_indiv) a.indiv[g] = r;
            if (has_done) a.done[g] = (uint8_t)(has_step ? (stp >= a.world_length) : 0);
            if (i == 0 && env_bad && a.nan_flag) a.nan_flag[e] = 1;         // the reference's failure mode (Q9), sticky
            if (i == 0 && has_step) {
                const T ret = epr + (T)R;                                   // epr == 0 when ep_return is not tracked
                const int ec = epc + coltot;
                epr = (!has_epr || (dn && a.auto_reset)) ? (T)0 : ret;
                epc = (!has_epc || (dn && a.auto_reset)) ? 0 : ec;
                if (has_epr) a.ep_return[e] = epr;
                if (has_epc) a.ep_coll[e] = epc;
                if (dn && has_stats) {
                    atomicAdd(&s_stat[0], 1.0);
                    atomicAdd(&s_stat[1], (double)ret);
                    atomicAdd(&s_stat[2], (double)ret * (double)ret);
                    atomicAdd(&s_stat[3], (double)ec);
                }
            }
        }

        // the reward hook's side effect (formation_hd_obs_env.py:85-88): every obstacle falls at (0, -1) while it is above
        // the floor and rests below it -- its velocity for the next step
        if (obst_lane) ov = O::make((T)0, (s_on[le * NO + i].y > a.ofloor) ? a.ofall : (T)0);

        // ======== VecEnv auto-reset (env_wrappers.py:14-18; reset_world formation_hd_partial_env.py:89-101)
        if (a.auto_reset && __any_sync(FULL, dn)) {
            const uint32_t tk = tick0 + (uint32_t)ts;
            if (dn) {
                if constexpr (EXT) {                                        // terminal block: the post-step state
                    if (a.fin_pos) {
                        a.fin_pos[g] = p; a.fin_vel[g] = v;
#pragma unroll
                        for (int k0 = 0; k0 < LG; k0 += N)
                            if (k0 + i < LG) a.fin_lm[(size_t)e * L + k0 + i] = s_lm[le * L + k0 + i];
                        if (OBST && i < NO) a.fin_lm[(size_t)e * L + LG + i] = s_on[le * NO + i];
                    }
                }
                U4 r = philox(a.seed, ge, (uint32_t)i, tk, kResetAgent);
                p = O::make(uniform_pm1<T>(r.x), uniform_pm1<T>(r.y));
                v = zero;
                s_pnew[le * 2 * N + i] = p;
                s_pnew[le * 2 * N + N + i] = p;
                s_vel[lane] = v;
                stp = 0;
#pragma unroll
                for (int k0 = 0; k0 < LG; k0 += N) {                        // landmarks i, i + N, ... of my env
                    const int k = k0 + i;
                    if (k < LG) {
                        U4 q = philox(a.seed, ge, (uint32_t)k, tk, kResetLandmark);
                        const R2 l = O::make(uniform_pm1<T>(q.x), uniform_pm1<T>(q.y));
                        s_lm[le * L + k] = l;
                        a.lm[(size_t)e * L + k] = l;
                    }
                }
                if (OBST && i < NO) {                                       // formation_hd_obs_env.py:108,116-119
                    R2 po;
                    obstacle_reset<T>(a.seed, ge, LG + i, i, NO, tk, &po, &ov, a.ofall);
                    s_on[le * NO + i] = po;
                }
                if (ts == n_steps - 1) { a.pos[g] = p; a.vel[g] = v; }
            }
            __syncwarp();
        }
        if (active && i == 0 && has_step) a.step[e] = stp;
        if (obst_lane && ts == n_steps - 1) {                               // the obstacles' new state
            a.lm[(size_t)e * L + LG + i] = s_on[le * NO + i];
            if (a.lmv) a.lmv[(size_t)e * L + LG + i] = ov;
        }

        // ================= observation rows leave the SM as one bulk copy =======================
        // Filled LAST, from the shared state, which for an env that was just reset already holds the RESET state
        // (env_wrappers.py:16-17): one code path writes both kinds of observation, and the bulk copy of the
        // previous span / step has had this whole step to finish reading the image.
        {
            if (bulk_pending) {
                if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                bulk_pending = false;
                __syncwarp();
            }
            // comm of the others (silent agents: zeros): nothing else writes these slots and the warp's spans all use the
            // same image (one 16-byte phase per warp), so they are written once per launch, not once per span
            if (zeroed != s_obs) {                                          // warp-uniform
                if (lane < NA) {
#pragma unroll
                    for (int m = 0; m < N - 1; ++m) s_obs[lane * IPR + 1 + L + NREL + m] = zero;
                }
                zeroed = s_obs;
            }
            // EVEN row stride: the landmark segment of all rows of the span is written by consecutive lanes <-> consecutive
            // (row, k) items -- the N rows of an env read the same L landmark items (broadcasts) and a half-warp's stores
            // fall on consecutive banks; "lane l writes item kk of its own row" has 2-way conflicts even in rotated
            // order (fg_warp.cuh, COOP_SHAPE: N = 4 29.6 -> 27.6 us there)
            // (not for the obstacle scenario: its relative obstacle entries need the row's agent as well, and the unrolled
            // loop then spills 72-112 bytes under the 80-register bound)
            constexpr bool COOP_LM = (IPR % 2) == 0 && !OBST;
            if constexpr (COOP_LM) {
#pragma unroll
                for (int it = 0; it < (NA * L + 31) / 32; ++it) {
                    const int q = it * 32 + lane;
                    if (q < NA * L) {
                        const int R = q / L, k = q - R * L;                 // row of the span, landmark
                        s_obs[R * IPR + 1 + k] = s_lm[(R / N) * L + k];     // landmark p_pos, absolute
                    }
                }
            }
            if (active) {
                // [p_vel | landmark p_pos (L) | other_pos (NREL) | comm of the others (N-1 zeros)]
                // (formation_hd_partial_env.py:40-65 / formation_hd_partial_range_env.py:40-54).  Own row per lane; an
                // EVEN row stride would put "item k of every row" on 32 / gcd(2 IPR, 32) banks, so each lane then walks
                // every row segment in an order rotated by its lane index (as fg_warp.cuh does for even N).
                constexpr bool ROT = (IPR % 2) == 0;
                R2* row = s_obs + lane * IPR;
                const R2* eL = s_lm + le * L;
                const R2* eP = s_pnew + le * 2 * N + i;                     // eP[k] = agent (i + k) mod N
                const R2* eA = s_pnew + le * 2 * N;                         // eA[j] = agent j
                row[0] = v;
                if constexpr (!COOP_LM) {
                    const int rL = ROT ? lane % L : 0;
#pragma unroll
                    for (int k = 0; k < L; ++k) {
                        int kk = k + rL; kk -= (kk >= L) ? L : 0;
                        R2 l = eL[kk];                                      // landmark p_pos, absolute
                        if (OBST && kk >= LG) {                             // obstacles: NEW position relative to me (:58-59)
                            const R2 o = s_on[le * NO + (kk - LG)];
                            l = O::make(O::sub(o.x, p.x), O::sub(o.y, p.y));
                        }
                        row[1 + kk] = l;
                    }
                }
                const int rR = ROT ? lane % NREL : 0;
#pragma unroll
                for (int m = 0; m < NREL; ++m) {
                    int mm = m + rR; mm -= (mm >= NREL) ? NREL : 0;
                    if (SCN == kScnPartial) {                               // agents i+1 .. i+NOBS, cyclic (:50-53)
                        R2 q = eP[1 + mm];
                        row[1 + L + mm] = O::make(O::sub(q.x, p.x), O::sub(q.y, p.y));
                    } else {                                                // all others, j != i ascending
                        R2 q = eA[mm + (mm >= i ? 1 : 0)];
                        T dx = O::sub(q.x, p.x), dy = O::sub(q.y, p.y);
                        if (SCN == kScnRange) {                             // clipped to the sensing range (:49-52)
                            const T lo = -a.obs_range, hi = a.obs_range;    // np.clip keeps NaN
                            dx = (dx < lo) ? lo : ((dx > hi) ? hi : dx);
                            dy = (dy < lo) ? lo : ((dy > hi) ? hi : dy);
                        }
                        row[1 + L + mm] = O::make(dx, dy);
                    }
                }
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");    // generic-proxy writes -> async proxy
            __syncwarp();
            const uint32_t head = obs_head < obs_bytes ? obs_head : obs_bytes;
            const uint32_t mid = (obs_bytes - head) & ~15u;
            const uint32_t tail = obs_bytes - head - mid;                   // 0 or 8 (fp32)
            if (lane == 0) {
                if (mid) {
                    uint64_t pol;                                           // write-once streaming output (fg_warp.cuh)
                    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
                    asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;"
                                 :: "l"(reinterpret_cast<unsigned char*>(g_obs) + head),
                                    "r"(smem_u32(reinterpret_cast<unsigned char*>(s_obs) + head)), "r"(mid), "l"(pol)
                                 : "memory");
                    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                }
            } else if (lane == 1) {
                if (head) g_obs[0] = s_obs[0];
            } else if (lane == 2) {
                if (tail) {
                    const uint32_t it = (head + mid) / (uint32_t)sizeof(R2);
                    g_obs[it] = s_obs[it];
                }
            }
            bulk_pending = true;
        }
        // next step of an in-kernel rollout: the obstacles' new positions become the old ones
        if (OBST && n_steps > 1 && obst_lane) s_lm[le * L + LG + i] = s_on[le * NO + i];
    }
    if (--spans_left == 0) break;
  }  // spans
    // the shared-memory image must outlive the bulk copy's reads
    if (bulk_pending && lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    __syncwarp();
    if (has_stats && lane < 4 && s_stat[0] != 0.0) atomicAdd(&a.stats[lane], s_stat[lane]);
    tick_arrive(a.tick_dev, (unsigned)min(nwarps, nspans), n_steps, lane == 0);
}

}  // namespace fg
