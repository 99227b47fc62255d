// fg_warp.cuh -- warp-autonomous fused step kernel for formation_hd_env with small N (sm_100a).
//
// Why it exists: at N = 9 the tile kernel in fg_kernels.cuh is ISSUE-bound, not HBM-bound
// (profiles/r01_baseline_*: 115 M warp instructions per 131072-env launch, 73 % issue-active, 28 %
// of the HBM roofline): it decodes (row, item) for every 8-byte observation item and crosses six
// CTA barriers per step.  This kernel removes both costs:
//
//   * N is a template constant and EPW = floor(32 / N) whole envs live in ONE warp (lane <-> agent),
//     so every exchange inside an env is warp-local: shared-memory slices private to the warp,
//     __syncwarp() only, no __syncthreads() anywhere.  Warps drift freely, which spreads their
//     load / compute / store phases over time.
//   * every pair loop is unrolled with compile-time shared-memory offsets; far pairs cost
//     6-7 instructions (a near-pair BITMASK is built branch-free and the softplus contact force /
//     the exact collision test run afterwards only for set bits, in ascending-j order = the
//     reference's accumulation order, core.py:242-254).
//   * each lane writes ITS OWN observation row (3N float2 items, compile-time offsets, conflict-free
//     because the row stride 3N is odd) into the warp's slice of shared memory, and the slice --
//     one contiguous span of the [E,N,6N] tensor -- leaves the SM as ONE TMA bulk store
//     (cp.async.bulk.global.shared::cta; SASS UBLKCP) issued by lane 0.  Row and env spans are only
//     8-byte aligned for odd N (fp32), so a span that starts/ends on an odd 8-byte slot sends that
//     one head/tail item with a plain 8-byte store.
//
// Semantics are those of fg::k_step<T, hd, PHYS, OBSREW> (fg_kernels.cuh) restricted to: uniform
// agent constants, no walls, silent agents, landmarks not tracked.  Everything else takes the
// tile kernel.  Reference citations are on the code below.
#pragma once
#include "fg_kernels.cuh"
#include "fg_policy.cuh"

namespace fg {

// log_NF(N) when N is a power of NF, else 0 (the shapes get_action_BFS accepts, formation_gym/__init__.py:55-56)
template <int N, int NF> struct PolLevels {
    static constexpr int v = (NF >= 2 && N > 1 && N % NF == 0 && (N == NF || PolLevels<N / (NF >= 2 ? NF : 2), NF>::v > 0))
                             ? 1 + PolLevels<N / (NF >= 2 ? NF : 2), NF>::v : 0;
};
template <int NF> struct PolLevels<1, NF> { static constexpr int v = 0; };
template <int NF> struct PolLevels<0, NF> { static constexpr int v = 0; };

// Per-warp shared-memory slice layout (bytes), shared by host (sizing) and device (carving).
template <typename T, int N, bool WOBS> struct WarpLayout {
    typedef typename Ops<T>::R2 R2;
    typedef typename Ops<T>::Bits Bits;
    static constexpr int EPW = 32 / N;             // envs per warp
    // Warps per CTA the kernel is compiled for.  N = 27 holds a 17.5 KB observation image per warp, so
    // shared memory caps the SM at 12 warps anyway: 4-warp CTAs let ptxas use up to 255 registers (with
    // 256-thread bounds it stopped at 128 and spilled two, and with ~2 KB of L1 left beside the shared
    // memory every spill reload went to L2 -- 34 % of all stall samples in profiles/r01c_warp27_before).
    // (N = 9 as seven 4-warp CTAs per SM -- 72 registers, no spills, 28 instead of 24 warps -- is no faster: 51.3 vs
    // 50.9 us at the burst clock, 55.7-56.2 vs 55.3-56.0 us after 1 s under load, 544 vs 521 us per 1 M envs.  Neither
    // more warps nor fewer instructions move the power-capped number, so it is not SM-side latency that follows the clock.)
    static constexpr int MAXW = (N >= 16) ? 4 : 8;
    static constexpr int MINB = (N >= 16) ? 0 : 3;
    // Where the observation image is filled.  LATE (after rewards / auto-reset, from the shared state):
    // the bulk copy of the previous span has the whole step to finish reading the image, at the price of
    // re-reading the partner positions (measured: N = 3 91.1 -> 86.9 us per 1 M envs, N = 27 246 -> 241 us
    // per 65536).  FUSED into the reward loop (the p_j - p_i it already holds): fewest instructions, best
    // where the kernel is closest to issue-bound (N = 9: 55.0 us fused vs 58.5 us late per 131072 envs).
    // (A/B build -DFG_LATE9=1, round 2 with the STD instantiation: late fill at N = 9 is now a tie -- 51.2 vs 52.2 us
    // L2-resident, 529.5 vs 530.2 us per 1 M envs -- so neither variant is what holds the streaming regime at 4.85 TB/s.)
#ifndef FG_LATE9
#define FG_LATE9 0
#endif
    static constexpr bool LATE_FILL = (N != 9) || FG_LATE9;   // N = 3, 9: three 8-warp CTAs per SM (<= 85 registers)
    static constexpr int NA = EPW * N;             // active lanes
    static constexpr int IPR = 3 * N;              // R2 items per observation row (6N scalars)
    static constexpr int OBS_ITEMS = WOBS ? NA * IPR : 0;
    static constexpr size_t off_obs = 0;                                     // +16 B slack for the 8-byte phase
    static constexpr size_t off_pold = off_obs + (WOBS ? (size_t)OBS_ITEMS * sizeof(R2) + 16 : 0);
    static constexpr size_t off_pnew = off_pold + (size_t)NA * sizeof(R2);   // [EPW][2N]: p_0..p_{N-1} twice
    static constexpr size_t off_cen = off_pnew + (size_t)2 * NA * sizeof(R2);
    static constexpr size_t off_shp = off_cen + (size_t)NA * sizeof(R2);
    static constexpr size_t off_vel = off_shp + (size_t)NA * sizeof(R2);
    static constexpr size_t off_mean = off_vel + (size_t)NA * sizeof(R2);    // [EPW][2]: mean pos, mean vel
    static constexpr size_t off_max = off_mean + (size_t)2 * EPW * sizeof(R2);
    static constexpr size_t off_col = off_max + (size_t)EPW * sizeof(Bits);
    static constexpr size_t off_stat = (off_col + (size_t)EPW * sizeof(int) + 7) & ~(size_t)7;   // 4 doubles
    static constexpr size_t raw = off_stat + 4 * sizeof(double);
    static constexpr size_t stride = (raw + 15) & ~(size_t)15;
};

// SCN == kScnBasic (basic_formation_env with L == N landmarks, e.g. the default 3 agents / 3 landmarks): the same
// kernel with lane i doubling as landmark i -- the landmark rides in the `S` slot of the ideal shape, the reward is
// -sum_k min_a |p_a - l_k| - #{a incl. self : |p_a - p_i| < s_a + s_i} (basic_formation_env.py:43-52), the row is
// [p_vel, p_pos, l_k - p, p_j - p, comm] (basic_formation_env.py:29-41; also 3N items when L == N).
//
// STD (fp32 only): the standard product configuration, asserted by the host before it picks this instantiation --
// agents collide, unit mass, no max_speed, one step per launch, the step / done / indiv / ep_return /
// ep_collisions / stats buffers present and no comm buffer (silent agents: c == 0).  Each of these is otherwise a
// warp-uniform run-time test (constant load + compare + branch, plus a reconvergence pair inside divergent code):
// at N = 3 such tests were a fifth of the 61 instructions per env-step (profiles/r02b_warp3: ISETP 11.6 %, BRA 7.3 %,
// LDCU 6.4 %, BSSY/BSYNC 7 % of all warp instructions).
//
// POL > 0 (formation_hd_env, N = POL^k): the reference's demo controller get_action_BFS(ezpolicy, obs_n, POL)
// (formation_gym/__init__.py:19-98; test.py:23) runs on the NEW state at the end of every step -- the state the
// observations just returned describe, i.e. the reset state for an env whose episode ended -- and its actions are
// written to the action buffer for the NEXT step (and carried in registers between the steps of a rollout).  The
// positions, the ideal shape and ideal_vel are already on chip, so the controller costs its arithmetic only: no second
// launch, no re-read of the state (fg_policy.cuh: policy_chain; each lane evaluates the nodes of its own leaders).
//
// EXT (reset extension): the auto-reset takes the env's task from the target bank (KArgs::tgt_*, formation_hd_env) and
// copies the terminal state into the terminal block (KArgs::fin_*), each when set (run-time tests).  A separate
// instantiation: the reset block shares the registers of the step, and a bank branch compiled into every kernel changed
// the allocation (and added spills) of the product instantiations.
template <typename T, int N, bool WOBS, int SCN = kScnHD, bool STD = false, int POL = 0, bool EXT = false>
// (basic_formation_env, N = 3: four 8-warp CTAs per SM -- 64 registers, no spills -- measured 80.9 vs 88.7 us per 1 M envs;
// the hd instantiation of the same N loses with them: 89.2 vs 82.0 us)
__global__ void __launch_bounds__(32 * WarpLayout<T, N, WOBS>::MAXW, (SCN == kScnBasic && sizeof(T) == 4) ? 4 : WarpLayout<T, N, WOBS>::MINB) k_hd_warp(const __grid_constant__ KArgs<T> a) {
    static_assert(SCN == kScnHD || WarpLayout<T, N, WOBS>::LATE_FILL, "basic rows are written by the late fill");
    static_assert(POL == 0 || (SCN == kScnHD && PolLevels<N, POL>::v > 0), "POL: formation_hd_env with N = POL^k agents");
    typedef Ops<T> O;
    typedef typename O::R2 R2;
    typedef typename O::Bits Bits;
    typedef WarpLayout<T, N, WOBS> LY;
    constexpr int EPW = LY::EPW, NA = LY::NA, IPR = LY::IPR;
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
    const unsigned envmask = (N == 32 ? 0xffffffffu : ((1u << (N & 31)) - 1u)) << (le * N);   // lanes of this env

    unsigned char* wr = smem_raw + (size_t)wib * LY::stride;
    R2* s_pold = reinterpret_cast<R2*>(wr + LY::off_pold);
    R2* s_pnew = reinterpret_cast<R2*>(wr + LY::off_pnew);
    R2* s_cen = reinterpret_cast<R2*>(wr + LY::off_cen);
    R2* s_shp = reinterpret_cast<R2*>(wr + LY::off_shp);
    R2* s_vel = reinterpret_cast<R2*>(wr + LY::off_vel);
    R2* s_mean = reinterpret_cast<R2*>(wr + LY::off_mean);
    Bits* s_max = reinterpret_cast<Bits*>(wr + LY::off_max);
    int* s_col = reinterpret_cast<int*>(wr + LY::off_col);
    // episode statistics of this warp's envs: accumulated here (shared-memory atomics, episode ends
    // only) and sent to HBM as ONE set of 4 atomics per warp when the kernel ends -- per-env global
    // atomics on 4 addresses serialise in L2 (measured: 0.75 ms per episode end at 131072 envs).
    double* s_stat = reinterpret_cast<double*>(wr + LY::off_stat);
    if (lane < 4) s_stat[lane] = 0.0;

    // Shared-memory image of the span's observation rows.  It starts at the same offset modulo 16
    // as the span does in HBM so that the 16-byte-aligned middle can leave as one bulk copy; with
    // an even warp stride that phase is the same for every span of this warp.
    // (recomputed per span from the span's address -- cheaper than keeping it live across the loop)

    const R2 zero = O::make((T)0, (T)0);
    bool bulk_pending = false;
    // ZERO_ONCE: the comm slots of the row image (N - 1 zeros per row: silent agents) are written once per launch --
    // nothing else writes them and every span of a warp uses the same image position (one 16-byte phase per warp, see
    // the host).  Per N by measurement (same box, us per step, rewritten every span -> once): N = 4 30.4 -> 29.7,
    // 6 59.9 -> 57.1, 7 34.7 -> 34.3, 8 45.6 -> 44.6, 25 230.0 -> 192.3; but 9 51.9 -> 53.1, 16 77.3 -> 83.5,
    // 27 209.5 -> 236.5, 32 151.5 -> 158.0 (the fill is no longer the same instruction stream in every span and the
    // schedule ptxas finds is worse), so those keep the stores.
    constexpr bool ZERO_ONCE = (N >= 4 && N <= 8) || N == 25;
    bool comm_zeroed = false;

    // Software pipeline over the spans of this (persistent) warp: the state of span s + nwarps is
    // requested from HBM before span s is computed, so the load latency hides behind ~800
    // instructions of work instead of stalling the warp.
    R2 p_n = zero, v_n = zero, u_n = zero, S_n = zero, iv_n = zero;
    T epr_n = (T)0;
    int stp_n = 0, epc_n = 0;
    auto fetch = [&](int span) {
        const int fe0 = span * EPW;
        const bool act = lane < min(EPW, a.E - fe0) * N;
        p_n = zero; v_n = zero; u_n = zero; S_n = zero; iv_n = zero; stp_n = 0; epr_n = (T)0; epc_n = 0;
        if (act) {                                                          // coalesced: lane <-> consecutive agent
            const size_t fa = (size_t)fe0 * N + lane;
            p_n = a.pos[fa];
            v_n = a.vel[fa];
            if (SCN == kScnBasic) S_n = a.lm[fa];                          // landmark `lane` of the span (L == N)
            else { S_n = a.shape[fa]; iv_n = a.ivel[fe0 + le]; }
            if (!a.random_actions) u_n = a.act[fa];
            if (has_step) stp_n = a.step[fe0 + le];
            if (i == 0) {                                                   // running episode statistics of the env
                if (has_epr) epr_n = a.ep_return[fe0 + le];
                if (has_epc) epc_n = a.ep_coll[fe0 + le];
            }
        }
    };
    // L2 prefetch of the span AFTER the one `fetch` requests (two iterations ahead of the one being computed).  Once the
    // state arrays no longer fit in the 126 MB L2 (E >~ 200 K envs at N = 9) a register prefetch one iteration ahead
    // is not enough: under the write-saturated DRAM queues a read takes longer than the ~4 us of one iteration
    // (profiles/r02b_warp9_e1M: long-scoreboard stalls 3.2 per issue on the first use of the prefetched registers,
    // 4.7 TB/s of DRAM traffic against 6.0 when the state is L2-resident).  prefetch.global.L2 costs no registers
    // and no shared memory; the register prefetch of the next iteration then hits in L2.
    auto l2_prefetch = [&](int span) {
        const int fe0 = span * EPW;
        if (fe0 >= a.E) return;                                             // warp-uniform
        // One request per 128-byte line: a span's chunk of an array is NA * 8 <= 256 bytes, so the lines holding its
        // first element, its 17th (+128 B) and its last one cover it.  (A prefetch per lane was measured 10 % SLOWER at
        // N = 9 with an L2-resident state -- 108 requests per iteration; testing every lane's address for a line start
        // cost 9 % of the instructions at N = 3; bulk TMA prefetches, one per array, were worse still: they queue with
        // the observation bulk store.)
        const int nact = min(EPW, a.E - fe0) * N;
        if ((lane == 0 || lane == 16 || lane == nact - 1) && lane < nact) {
            const size_t fa = (size_t)fe0 * N + lane;
            asm volatile("prefetch.global.L2 [%0];" :: "l"(a.pos + fa));
            asm volatile("prefetch.global.L2 [%0];" :: "l"(a.vel + fa));
            asm volatile("prefetch.global.L2 [%0];" :: "l"((SCN == kScnBasic ? a.lm : a.shape) + fa));
            if (!a.random_actions) asm volatile("prefetch.global.L2 [%0];" :: "l"(a.act + fa));
        }
    };
    fetch(gw);
    for (int d = 1; d < a.pf_dist; ++d) l2_prefetch(gw + d * nwarps);

  int spans_left = (nspans - gw + nwarps - 1) / nwarps;                     // >= 1
  for (int span = gw; ; span += nwarps) {
    const int env0 = span * EPW;
    const int nval = min(EPW, a.E - env0);
    const bool active = lane < nval * N;
    const int e = env0 + le;
    const size_t g = (size_t)env0 * N + lane;                               // global agent index
    const uint32_t ge = a.env_offset + (uint32_t)e;                         // global env id (Philox counter)
    R2* g_obs = WOBS ? a.obs + (size_t)env0 * N * IPR : nullptr;
    const uint32_t obs_bytes = WOBS ? (uint32_t)(nval * N * IPR) * (uint32_t)sizeof(R2) : 0u;
    const uint32_t obs_head = WOBS ? (uint32_t)((16u - ((uint32_t)(uintptr_t)g_obs & 15u)) & 15u) : 0u;   // 0 or 8 (fp32), 0 (fp64)
    R2* s_obs = WOBS ? reinterpret_cast<R2*>(wr + LY::off_obs + ((16u - obs_head) & 15u)) : nullptr;

    R2 p = p_n, v = v_n, u = u_n, S = S_n, iv = iv_n;
    T epr = epr_n;
    int stp = stp_n, epc = epc_n;
    if (spans_left > 1) fetch(span + nwarps);
    if (a.pf_dist > 0 && spans_left > a.pf_dist) l2_prefetch(span + a.pf_dist * nwarps);
    __syncwarp();                                                           // previous span's readers of s_shp are done
    if (lane < NA) s_shp[lane] = S;

    for (int ts = 0; ts < n_steps; ++ts) {
        if (lane < EPW) { s_max[lane] = 0; s_col[lane] = 0; }
        if (lane < NA) s_pold[lane] = p;
        // Does my env hold a non-finite old position?  Then every pair goes to the contact force (env_cut2,
        // fg_kernels.cuh).  The warp-uniform vote on |x| + |y| (inactive lanes hold zeros) keeps the common path at a few
        // instructions; the exact per-env ballot runs only in a warp that has such a position (or one near FLT_MAX).
        const bool warp_nf = f_collide && __any_sync(FULL, !(fabs(p.x) + fabs(p.y) < (T)INFINITY));
        bool env_nf = false;
        if (warp_nf) env_nf = (__ballot_sync(FULL, active && nonfinite2(p.x, p.y)) & envmask) != 0u;
        __syncwarp();

        // =============================== World.step (core.py:206-225) ===========================
        if (active) {
            // (Round 2: an instantiation that draws the NEXT span's actions inside the reward / row-fill block -- the
            // Philox chain interleaved with shared-memory waits instead of standing here in a block of its own -- is
            // bit-identical and a tie: N = 9 57.4 vs 56.7 us, N = 27 220.7 vs 220.7, N = 3 93.8 vs 95.2, N = 16 74.0
            // vs 74.8, same box after 1 s under load.  The draw is not on the critical path; not kept.)
            if (a.random_actions) {                                         // test.py:20
                U4 r = philox(a.seed, ge, (uint32_t)i, tick0 + (uint32_t)ts, kAction);
                u = O::make(uniform_pm1<T>(r.x), uniform_pm1<T>(r.y));
                if (a.random_actions == 2) const_cast<R2*>(a.act)[g] = u;   // recorded for the caller (replay buffer)
            }
            // _set_action: u *= sensitivity (environment.py:216-221); apply_action_force:
            // F = gain * u + noise (core.py:232-236)
            T Fx = O::mul(a.gain, O::mul(u.x, a.sens));
            T Fy = O::mul(a.gain, O::mul(u.y, a.sens));
            if (f_noise) {
                U4 r = philox(a.seed, ge, (uint32_t)i, tick0 + (uint32_t)ts, kUNoise);
                T n0, n1; normal_pair<T>(r.x, r.y, &n0, &n1);
                Fx = O::add(Fx, O::mul(n0, a.u_noise));
                Fy = O::add(Fy, O::mul(n1, a.u_noise));
            }
            // apply_environment_force (core.py:240-254).  Pass 1 (branch-free, unrolled): bit j of
            // `near` <=> pair (i, j) is inside the contact cut-off (or its distance is NaN).
            if (f_collide) {
                const R2* ep = s_pold + le * N;
                unsigned near = 0;
#pragma unroll
                for (int j = 0; j < N; ++j) {
                    R2 q = ep[j];
                    T dx = O::sub(p.x, q.x), dy = O::sub(p.y, q.y);
                    T d2 = dx * dx + dy * dy;
                    near |= (!(d2 >= a.cut2)) ? (1u << j) : 0u;             // !(>=) keeps NaN pairs
                }
                if (warp_nf && env_nf) near = (N == 32) ? 0xffffffffu : ((1u << (N & 31)) - 1u);   // and inf ones
                near &= ~(1u << i);
                // (Round 2: the point differences of this loop and of the reward loop as ONE packed FMA each --
                // fma.rn.f32x2 p * (-1, -1) + q, bit-identical to two FSUBs, 35 FFMA2 and 40 fewer SASS instructions at
                // N = 9 -- is a tie on a box that holds 1965 MHz: N = 9 50.95 vs 50.85 us, N = 16 78.0 vs 75.8, N = 25
                // 188.4 vs 192.0, N = 3 82.2 vs 81.6; and after 1 s under load (clock under the power cap): N = 9 54.5 vs
                // 54.4-54.8, N = 16 79.2 vs 71.6.  Not kept.)
                // Pass 2: the near pairs in ascending j -- the order in which the reference's a<b
                // double loop adds contributions to agent i.
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
            }
            // integrate_state (core.py:264-277); F / m with m == 1 is exact, skip the division
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
            // update_agent_state (core.py:279-286): silent agents -> c = 0
            s_pnew[le * 2 * N + i] = p;
            s_pnew[le * 2 * N + N + i] = p;
            s_vel[lane] = v;
            if (ts == n_steps - 1) {
                a.pos[g] = p; a.vel[g] = v;
                if (has_comm) a.comm[g] = zero;
            }
        }
        // any non-finite position in an env makes its centroid, hence the whole shape term, NaN
        const bool bad = !(fabs(p.x) < (T)INFINITY) || !(fabs(p.y) < (T)INFINITY);
        const bool env_bad = (__ballot_sync(FULL, active && bad) & envmask) != 0u;
        __syncwarp();

        // ================= Scenario.reward on the NEW state (formation_hd_env.py:61-75; Q16) =====
        // centroid and mean velocity: one lane per (env, {pos, vel}), summed in agent order like
        // np.mean(axis=0)
        if (SCN == kScnHD && lane < 2 * nval) {
            const int qe = lane >> 1, which = lane & 1;
            const R2* src = which ? (s_vel + qe * N) : (s_pnew + qe * 2 * N);
            T sx = 0, sy = 0;
#pragma unroll
            for (int j = 0; j < N; ++j) { R2 q = src[j]; sx = O::add(sx, q.x); sy = O::add(sy, q.y); }
            s_mean[lane] = O::make(O::div_count(sx, N), O::div_count(sy, N));   // np.mean: fp64 divides, fp32 multiplies by 1/N
        }
        __syncwarp();
        const R2 mp = (SCN == kScnHD) ? s_mean[2 * le] : zero, mv = (SCN == kScnHD) ? s_mean[2 * le + 1] : zero;
        const R2 C = O::make(O::sub(p.x, mp.x), O::sub(p.y, mp.y));         // centred agent shape
        if (SCN == kScnHD && lane < NA) s_cen[lane] = C;
        if (WOBS && !LY::LATE_FILL && bulk_pending) {                       // previous image is still being read
            if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
            bulk_pending = false;
        }
        __syncwarp();

        int col = 0;
        if (SCN == kScnBasic) {
            T* s_lmin = reinterpret_cast<T*>(s_cen);                        // [NA] min_a |p_a - l_k| per landmark
            if (active) {
                const R2* eA = s_pnew + le * 2 * N;                         // eA[k] = agent k
                // reward part 1 (basic_formation_env.py:45-47), lane i <-> landmark i = S
                T m = (T)INFINITY;                                          // min_a |p_a - l|^2; one sqrt after the loop
                bool nan_seen = false;
                unsigned hit = 0;
#pragma unroll
                for (int k = 0; k < N; ++k) {
                    R2 q = eA[k];
                    T d = O::norm2sq(O::sub(q.x, S.x), O::sub(q.y, S.y));
                    nan_seen |= (d != d);
                    m = fmin(m, d);
                    // is_collision candidates, self included (basic_formation_env.py:48-51,89-91)
                    T dx = O::sub(q.x, p.x), dy = O::sub(q.y, p.y);
                    hit |= (dx * dx + dy * dy < a.rthr2_hi) ? (1u << k) : 0u;
                }
                s_lmin[lane] = nan_seen ? O::from_bits(~(Bits)0 >> 1) : O::sqrt_(m);
                while (f_collide && hit) {
                    const int k = __ffs(hit) - 1;
                    hit &= hit - 1;
                    R2 q = eA[k];
                    if (O::norm2(O::sub(q.x, p.x), O::sub(q.y, p.y)) < a.rthr) ++col;
                }
                if (col) atomicAdd(&s_col[le], col);
            }
        } else
        if (active) {
            const R2* eS = s_shp + le * N;
            const R2* eC = s_cen + le * N;
            const R2* eP = s_pnew + le * 2 * N + i;                         // eP[k] = agent (i + k) mod N
            constexpr bool FUSE = WOBS && !LY::LATE_FILL;
            R2* row = FUSE ? (s_obs + lane * IPR) : nullptr;
            T rowmin = (T)INFINITY, colmin = (T)INFINITY;
            unsigned hit = 0;
            if (FUSE) row[0] = v;                                           // p_vel
#pragma unroll
            for (int k = 0; k < N; ++k) {
                // symmetric Hausdorff partials (formation_hd_env.py:64-66): row i = min_k |C_i - S_k|^2,
                // column i = min_k |C_k - S_i|^2
                R2 Sk = eS[k], Ck = eC[k];
                rowmin = fmin(rowmin, O::sq2(O::sub(C.x, Sk.x), O::sub(C.y, Sk.y)));
                colmin = fmin(colmin, O::sq2(O::sub(Ck.x, S.x), O::sub(Ck.y, S.y)));
                if (FUSE) row[2 * N - 1 + k] = Sk;                          // ideal_shape.flatten()
                if (k >= 1) {
                    R2 q = eP[k];
                    T dx = O::sub(q.x, p.x), dy = O::sub(q.y, p.y);         // other_pos (formation_hd_env.py:55)
                    if (FUSE) {
                        // (a slot-ordered variant -- same store offset in every lane, partner index at run time --
                        // removes the 4-way store conflicts of this order but was measured slower at N = 9:
                        // 59.4 vs 53.6 us per 131072 envs)
                        const int slot = (i + k < N) ? (i + k) : (i + k - N + 1);
                        row[slot] = O::make(dx, dy);
                    }
                    T d2 = dx * dx + dy * dy;
                    hit |= (d2 < a.rthr2_hi) ? (1u << k) : 0u;
                }
            }
            if (FUSE) {
                if (!ZERO_ONCE || !comm_zeroed) {
#pragma unroll
                    for (int k = 0; k < N - 1; ++k) row[N + k] = zero;      // comm of the others (silent)
                }
                row[3 * N - 1] = iv;                                        // ideal_vel
            }
            // is_collision (formation_hd_env.py:71-74,119-121): exact test only for candidates
            while (f_collide && hit) {
                const int k = __ffs(hit) - 1;
                hit &= hit - 1;
                R2 q = eP[k];
                if (O::norm2(O::sub(q.x, p.x), O::sub(q.y, p.y)) < a.rthr) ++col;
            }
            atomicMax(&s_max[le], O::bits(fmax(rowmin, colmin)));           // d2 >= 0: bit order == value order
            if (col) atomicAdd(&s_col[le], col);
        }
        __syncwarp();

        // ============ rewards, done, statistics (environment.py:126-138,172-177) ================
        stp += 1;                                                           // environment.py:114
        const bool dn = active && has_step && (stp >= a.world_length);
        if (active) {
            T base;
            if (SCN == kScnBasic) {
                const T* s_lmin = reinterpret_cast<const T*>(s_cen) + le * N;
                base = (T)0;
#pragma unroll
                for (int k = 0; k < N; ++k) base = O::sub(base, s_lmin[k]);  // rew -= min(dists), landmark order
            } else {
                T form = -O::sqrt_(O::from_bits(s_max[le]));                // -max(dH(C,S), dH(S,C))
                if (env_bad) form = O::from_bits(~(Bits)0 >> 1);            // NaN, as the reference
                T velr = O::norm2(O::sub(iv.x, mv.x), O::sub(iv.y, mv.y));  // formation_hd_env.py:68-69
                base = O::sub(form, velr);
            }
            T r = base;
            for (int c = 0; c < col; ++c) r = O::sub(r, (T)1);              // rew -= 1 per collision
            const int coltot = s_col[le];
            // shared reward = sum_i r_i (environment.py:136): N*base - total collisions, in fp64
            const double R = (double)N * (double)base - (double)coltot;
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

        // ======== VecEnv auto-reset (env_wrappers.py:14-18; reset_world formation_hd_env.py:77-95)
        if (a.auto_reset && __any_sync(FULL, dn)) {
            const uint32_t tk = tick0 + (uint32_t)ts;
            R2 lraw = zero;
            if (dn) {
                if constexpr (EXT) {                                        // terminal block: the post-step state
                    if (a.fin_pos) {
                        a.fin_pos[g] = p; a.fin_vel[g] = v;
                        if (SCN == kScnBasic) a.fin_lm[g] = S;              // landmark `lane` of the span (L == N)
                        else { a.fin_shape[g] = S; if (i == 0) a.fin_ivel[e] = iv; }
                    }
                }
                U4 r = philox(a.seed, ge, (uint32_t)i, tk, kResetAgent);
                p = O::make(uniform_pm1<T>(r.x), uniform_pm1<T>(r.y));
                v = zero;
                U4 q = philox(a.seed, ge, (uint32_t)i, tk, kResetLandmark);
                lraw = O::make(uniform_pm1<T>(q.x), uniform_pm1<T>(q.y));
                s_pnew[le * 2 * N + i] = p;
                s_pnew[le * 2 * N + N + i] = p;
                stp = 0;
                if (SCN == kScnBasic) {                                     // basic_formation_env.py:54-65: no shape, no ideal_vel
                    S = lraw;
                    s_shp[lane] = S;
                    a.lm[g] = S;
                    if (ts == n_steps - 1) { a.pos[g] = p; a.vel[g] = v; }
                } else {
                    U4 w = philox(a.seed, ge, 0u, tk, kResetIdealVel);
                    iv = O::make(uniform_pm1<T>(w.x), uniform_pm1<T>(w.y));
                    if constexpr (EXT) {                                    // target bank: the task's shape / velocity
                        if (a.tgt_count > 0) {
                            const uint32_t kt = target_task<T>(a, e, ge, tk);
                            lraw = a.tgt_shape[(size_t)kt * N + i];
                            if (a.tgt_vel) iv = a.tgt_vel[kt];
                        }
                    }
                    s_pold[lane] = lraw;                                    // scratch: pold is dead until the next step
                    if (i == 0) a.ivel[e] = iv;
                }
            }
            __syncwarp();
            if (SCN == kScnHD && dn) {
                const R2* raw = s_pold + le * N;
                T sx = 0, sy = 0;
                for (int j = 0; j < N; ++j) { sx = O::add(sx, raw[j].x); sy = O::add(sy, raw[j].y); }
                S = O::make(O::sub(lraw.x, O::div(sx, (T)N)), O::sub(lraw.y, O::div(sy, (T)N)));   // :93
                s_shp[lane] = S;
                a.shape[g] = S;
                if (ts == n_steps - 1) { a.pos[g] = p; a.vel[g] = v; }
            }
            __syncwarp();
        }
        if (active && i == 0 && has_step) a.step[e] = stp;

        // ================= observation rows leave the SM as one bulk copy =======================
        // LATE_FILL: the image is filled LAST: the bulk copy of the previous span / step has had this whole step's
        // physics and reward to finish reading it (filling right after the physics left the warp waiting
        // on that copy for 25 % of its time at N = 27, profiles/r01c_warp27_before).  Rows come from the
        // shared state, which for an env that was just reset already holds the RESET state
        // (env_wrappers.py:16-17), so one code path writes both kinds of observation.
        if (WOBS) {
            if (bulk_pending) {
                if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                bulk_pending = false;
                __syncwarp();
            }
            // COOP_SHAPE (N = 4, 6, 8): the ideal_shape segment of all rows of the span is written by consecutive lanes <->
            // consecutive (row, k) items: the N rows of an env read the same N shape items (broadcasts) and a half-warp's
            // stores cover whole bank windows, where "lane l writes item kk of its own row" has 2-way conflicts even with
            // the rotated order (N = 4: 52 % of all shared-memory wavefronts were conflicts, the shape copy 13 % of the
            // stall samples: profiles/r02f_hd_n4)
            constexpr bool COOP_SHAPE = SCN == kScnHD && LY::LATE_FILL && (N == 4 || N == 6 || N == 8);
            if constexpr (COOP_SHAPE) {
#pragma unroll
                for (int it = 0; it < (NA * N + 31) / 32; ++it) {
                    const int q = it * 32 + lane;
                    if (q < NA * N) {
                        const int R = q / N, k = q - R * N;                 // row of the span, shape item
                        s_obs[R * IPR + 2 * N - 1 + k] = s_shp[(R / N) * N + k];
                    }
                }
            }
            if (LY::LATE_FILL ? active : dn) {                              // FUSED: only reset envs are rewritten
                // [p_vel | p_j - p_i (j != i ascending) | comm zeros | ideal_shape.flatten() | ideal_vel]
                // (formation_hd_env.py:52-59); own row per lane, odd row stride 3N -> conflict-free STS.64
                R2* row = s_obs + lane * IPR;
                const R2* eP = s_pnew + le * 2 * N + i;                     // eP[k] = agent (i + k) mod N
                const R2* eS = s_shp + le * N;
                row[0] = v;
                if constexpr (SCN == kScnHD && ((N & 1) == 0 || N >= 25)) {
                    // EVEN N: the row stride 3N items is a multiple of 8 (N = 4), 16 (N = 8) or 32 (N = 16) banks,
                    // so "every lane writes item k of its row" would hit 4 / 2 / 1 banks.  Each lane instead walks
                    // every row segment in an order rotated by its lane index (runtime indices, 2-3 way conflicts
                    // at worst): N = 16 173 -> see DESIGN.md.
                    const R2* eA = s_pnew + le * 2 * N;                     // eA[j] = agent j
                    const int r1 = lane % (N - 1), rN = lane % N;
#pragma unroll
                    for (int m = 0; m < N - 1; ++m) {
                        int mm = m + r1; mm -= (mm >= N - 1) ? (N - 1) : 0;
                        R2 q = eA[mm + (mm >= i ? 1 : 0)];                  // partner of slot mm: j != i ascending
                        row[1 + mm] = O::make(O::sub(q.x, p.x), O::sub(q.y, p.y));
                        if (!ZERO_ONCE) row[N + mm] = zero;                 // comm of the others (silent)
                    }
                    if (ZERO_ONCE && !comm_zeroed) {
#pragma unroll
                        for (int m = 0; m < N - 1; ++m) row[N + m] = zero;
                    }
                    // (writing the static 2N items of all rows cooperatively -- lane l holding items l, l + 32 of the
                    // env's [comm | ideal_shape | ideal_vel] vector, ceil(2N / 32) conflict-free stores per row -- was
                    // measured SLOWER at N = 27: 230.6 vs 209.1 us per 65536 envs; equal at N = 16, 25, 32)
                    if constexpr (!COOP_SHAPE) {
#pragma unroll
                        for (int k = 0; k < N; ++k) {
                            int kk = k + rN; kk -= (kk >= N) ? N : 0;
                            row[2 * N - 1 + kk] = eS[kk];
                        }
                    }
                    row[3 * N - 1] = iv;
                } else {
                // basic: [p_vel, p_pos, l_k - p (L = N), other_pos, comm] (basic_formation_env.py:29-41)
                constexpr int OFF = (SCN == kScnBasic) ? 1 + N : 0;         // other_pos starts at 1 + OFF
                if (SCN == kScnBasic) {
                    row[1] = p;
#pragma unroll
                    for (int k = 0; k < N; ++k) { R2 l = eS[k]; row[2 + k] = O::make(O::sub(l.x, p.x), O::sub(l.y, p.y)); }
                }
                const R2* eA = s_pnew + le * 2 * N;                         // eA[j] = agent j
#pragma unroll
                for (int m = 0; m < N - 1; ++m) {                           // slot order: same store offset in every lane
                    R2 q = eA[m + (m >= i ? 1 : 0)];
                    row[OFF + 1 + m] = O::make(O::sub(q.x, p.x), O::sub(q.y, p.y));   // other_pos (formation_hd_env.py:55)
                }
                if (!ZERO_ONCE || !comm_zeroed) {
#pragma unroll
                    for (int k = 0; k < N - 1; ++k) row[OFF + N + k] = zero;   // comm of the others (silent)
                }
                if (SCN == kScnHD) {
#pragma unroll
                    for (int k = 0; k < N; ++k) row[2 * N - 1 + k] = eS[k];
                    row[3 * N - 1] = iv;
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
                    // L2 evict_first: the rows are write-once streaming output; keeping them out of the
                    // way of the resident state arrays is worth 18 % at N = 9 (71.8 -> 58.9 us per step)
                    uint64_t pol;
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
            if (ZERO_ONCE) comm_zeroed = true;
        }

        // ====== device controller on the new state (formation_gym/__init__.py:49-98), under the bulk store ======
        if constexpr (POL > 0) {
            if (active) {
                u = policy_chain<T, POL, PolLevels<N, POL>::v>(s_pnew + le * 2 * N, s_shp + le * N, i, iv, a.pol_mult);
                if (ts == n_steps - 1) const_cast<R2*>(a.act)[g] = u;       // the next step's actions
            }
        }
    }
    if (--spans_left == 0) break;
  }  // spans
    // the shared-memory image must outlive the bulk copy's reads
    if (WOBS && bulk_pending && lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    __syncwarp();
    if (has_stats && lane < 4 && s_stat[0] != 0.0) atomicAdd(&a.stats[lane], s_stat[lane]);
    tick_arrive(a.tick_dev, (unsigned)min(nwarps, nspans), n_steps, lane == 0);
}

}  // namespace fg
