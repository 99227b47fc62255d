// fg_obstacle.cuh -- formation_hd_obs_env (formation_gym/envs/formation_hd_obs_env.py) on the tile layout of
// k_step: movable, colliding obstacle landmarks next to the agents and the (immovable, non-colliding) goal
// landmarks.
//
// Entity order of the reference's pair loop (core.py:143-144,240-254; formation_hd_obs_env.py:31-44):
// agents 0..N-1, goal landmarks (collide = False: every pair with them returns None, core.py:292), obstacles.
// Colliding pairs a < b are therefore agent-agent, agent-obstacle and obstacle-obstacle, all "both movable"
// (core.py:314-318).  Obstacles receive no action force, are damped and integrated like agents
// (core.py:264-277) and are never speed-clamped.  The scenario's reward hook rewrites every obstacle's velocity
// after the step: (0, -1) while it is above the floor y = -2.2, (0, 0) below (formation_hd_obs_env.py:85-88).
//
// One CTA owns EPC = floor(256 / N) envs; thread t <-> (local env, agent); obstacle and goal work is spread
// over the first threads (one per (env, obstacle) / (env, goal)).  `landmarks` is [E, L, 2] with the goals
// first and the O obstacles last; `landmark_vel` has the same shape (only obstacle entries are used).
#pragma once
#include "fg_kernels.cuh"

namespace fg {

constexpr int kScnObstacle = 4;     // formation_hd_obs_env

// Scenario.reset_world for obstacle k of O (formation_hd_obs_env.py:108,116-119): x ~ U(step[k], step[k+1]) with
// step = np.linspace(-1.8, 1.8, O + 1), y ~ U(2.0, 2.5), velocity (0, -1).  u01 on the 24-bit lattice.
template <typename T>
__device__ __forceinline__ void obstacle_reset(uint64_t seed, uint32_t ge, int slot, int k, int O, uint32_t tick,
                                               typename Ops<T>::R2* pos, typename Ops<T>::R2* vel, T fall_vy) {
    U4 r = philox(seed, ge, (uint32_t)slot, tick, kResetLandmark);
    const T u0 = (T)(r.x >> 8) * (T)(1.0 / 16777216.0), u1 = (T)(r.y >> 8) * (T)(1.0 / 16777216.0);
    const T w = (T)3.6 / (T)O;
    const T lo = (T)-1.8 + (T)k * w;
    const T hi = (k + 1 == O) ? (T)1.8 : (T)-1.8 + (T)(k + 1) * w;
    *pos = Ops<T>::make(lo + (hi - lo) * u0, (T)2.0 + (T)0.5 * u1);
    *vel = Ops<T>::make((T)0, fall_vy);
}

// OBSREW = false: World.step alone (core.py:206-225) on a world with obstacles -- no scenario hooks, so the
// obstacles keep their INTEGRATED velocity (the (0, -1) rule is the reward hook's side effect).
// EXT (reset extension, as in k_step): the auto-reset copies the terminal state into the terminal block (KArgs::fin_*).
// Without PHYS, EXT is fg_final_obs: the state is the terminal block, a CTA without an ended env (fin_done) exits at
// once, and no reward is written.
template <typename T, bool PHYS, bool OBSREW = true, bool EXT = false>
__global__ void __launch_bounds__(kBlock, 2) k_step_obst(const __grid_constant__ KArgs<T> a) {
    static_assert(PHYS || OBSREW, "nothing to do");
    typedef Ops<T> O_;
    typedef typename O_::R2 R2;
    typedef typename O_::Bits Bits;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr bool FINOBS = EXT && !PHYS;

    const int N = a.N, EPC = a.EPC, L = a.L, NO = a.n_obst, LG = a.L - a.n_obst;
    const int nA = EPC * N;
    R2* s_old = reinterpret_cast<R2*>(smem_raw);      // agent positions the contact force reads
    R2* s_new = s_old + nA;                           // after integration
    R2* s_v = s_new + nA;
    R2* s_cen = s_v + nA;                             // centred new positions
    R2* s_lm = s_cen + nA;                            // [EPC][L] goals, then obstacles (positions before the step)
    R2* s_on = s_lm + EPC * L;                        // [EPC][NO] obstacle positions after the step
    R2* s_ov = s_on + EPC * NO;                       // [EPC][NO] obstacle velocities
    R2* s_mean = s_ov + EPC * NO;                     // [EPC][2] agent centroid, goal centroid
    Bits* s_rowmax = reinterpret_cast<Bits*>(s_mean + 2 * EPC);
    int* s_col = reinterpret_cast<int*>(s_rowmax + EPC);
    int* s_dn = s_col + EPC;
    int* s_bad = s_dn + EPC;
    __shared__ double s_stat[4];
    if (threadIdx.x < 4) s_stat[threadIdx.x] = 0.0;

    const int t = threadIdx.x;
    const uint32_t tick0 = a.tick + (a.tick_dev ? a.tick_dev[0] : 0u);
    const int tile0 = blockIdx.x * EPC;
    const int le = (int)fastdiv((uint32_t)t, a.magic_n);
    const int i = t - le * N;
    const int e = tile0 + le;
    const bool active = (t < nA) && (e < a.E);
    const int nvalid = min(EPC, a.E - tile0);
    const size_t g = (size_t)e * N + i;
    const uint32_t ge = a.env_offset + (uint32_t)e;
    const T dmin_aa = O_::add(a.size, a.size);                    // core.py:307
    const T dmin_ao = O_::add(a.size, a.osize);
    const T dmin_oo = O_::add(a.osize, a.osize);
    const T cut_ao = dmin_ao + a.kcut * a.margin, cut_oo = dmin_oo + a.kcut * a.margin;
    const T cut2_ao = cut_ao * cut_ao, cut2_oo = cut_oo * cut_oo;

    // Gather mode (fg_obs_gather, as in k_step): slot e reads record gth_rows[e] with 64-bit addressing; a slot without
    // a record reads nothing and gets NaN state.
    long long rec = e;
    if constexpr (FINOBS) {
        if (a.gth_rows) {
            if (active) rec = gather_record(a, e);
        } else if (!__syncthreads_or(t < nvalid && a.fin_done[(size_t)(tile0 + t) * N] != 0)) {
            return;                                          // rows only where an episode ended (EPC <= kBlock)
        }
    }
    const R2 nan2 = O_::make((T)NAN, (T)NAN);

    R2 p = O_::make((T)0, (T)0), v = p, u = p;
    int stp = 0;
    if (active) {
        const size_t gs = FINOBS ? (size_t)rec * N + i : g;
        p = (FINOBS && rec < 0) ? nan2 : a.pos[gs];
        v = (FINOBS && rec < 0) ? nan2 : a.vel[gs];
        if (PHYS && !a.random_actions) u = a.act[g];
        if (PHYS) s_old[t] = p; else { s_new[t] = p; s_v[t] = v; }
        if (a.step) stp = a.step[e];
    }
    if (FINOBS && a.gth_rows) {                              // goals and obstacles of each slot's record
        for (int q = t; q < nvalid * L; q += kBlock) {
            const int qe = q / L, k = q - qe * L;
            const long long r = gather_record(a, tile0 + qe);
            const R2 l = r < 0 ? nan2 : a.lm[(size_t)r * L + k];
            s_lm[q] = l;
            if (k >= LG) { s_on[qe * NO + (k - LG)] = l; s_ov[qe * NO + (k - LG)] = O_::make((T)0, (T)0); }
        }
    } else {
        for (int q = t; q < nvalid * L; q += kBlock) s_lm[q] = a.lm[(size_t)tile0 * L + q];
        for (int q = t; q < nvalid * NO; q += kBlock) {
            const int qe = q / NO, k = q - qe * NO;
            const size_t gi = (size_t)(tile0 + qe) * L + LG + k;
            s_ov[q] = a.lmv ? a.lmv[gi] : O_::make((T)0, (T)0);
            if (!PHYS) s_on[q] = a.lm[gi];
        }
    }

    if (PHYS) __syncthreads();                               // the obstacle positions above, for the checks below

    for (int ts = 0; ts < a.n_steps; ++ts) {
        if (t < EPC) { s_rowmax[t] = 0; s_col[t] = 0; s_bad[t] = 0; }
        // some env of the tile holds a non-finite old agent or obstacle position: then every thread scans its env and
        // such an env runs with NaN contact cut-offs (env_cut2, fg_kernels.cuh).  Each check reads this thread's own
        // writes: s_old[t] (= p) and, for ts > 0, the obstacle entries of the stride loop at the end of the step.
        bool obad = false;
        if (PHYS) {                                           // (obstacle pairs collide whatever a.collide says)
            obad = active && nonfinite2(p.x, p.y);
            for (int q = t; q < nvalid * NO; q += kBlock) {
                const R2 po = s_lm[(q / NO) * L + LG + q % NO];
                obad |= nonfinite2(po.x, po.y);
            }
        }
        const bool tile_nf = __syncthreads_or(obad ? 1 : 0) != 0;
        auto env_nf = [&](int qe) -> bool {
            return tile_nf && (any_nonfinite(s_old + qe * N, N) || any_nonfinite(s_lm + qe * L + LG, NO));
        };

        // =============================== World.step (core.py:206-225) ===========================
        if (PHYS) {
            if (active) {
                if (a.random_actions) {
                    U4 r = philox(a.seed, ge, (uint32_t)i, tick0 + (uint32_t)ts, kAction);
                    u = O_::make(uniform_pm1<T>(r.x), uniform_pm1<T>(r.y));
                    if (a.random_actions == 2) const_cast<R2*>(a.act)[g] = u;    // recorded for the caller (replay buffer)
                }
                T Fx = O_::mul(a.gain, O_::mul(u.x, a.sens));                // environment.py:216-221, core.py:232-236
                T Fy = O_::mul(a.gain, O_::mul(u.y, a.sens));
                if (a.u_noise > (T)0) {
                    U4 r = philox(a.seed, ge, (uint32_t)i, tick0 + (uint32_t)ts, kUNoise);
                    T n0, n1; normal_pair<T>(r.x, r.y, &n0, &n1);
                    Fx = O_::add(Fx, O_::mul(n0, a.u_noise));
                    Fy = O_::add(Fy, O_::mul(n1, a.u_noise));
                }
                if (a.collide) {
                    const bool nf = env_nf(le);
                    const T c2_aa = env_cut2(a.cut2, nf), c2_ao = env_cut2(cut2_ao, nf);
                    // agent-agent pairs, other index ascending (equal masses: ratio 1)
                    const R2* envp = s_old + le * N;
                    for (int j = 0; j < N; ++j) {
                        if (j == i) continue;
                        R2 q = envp[j];
                        T dx = (j < i) ? O_::sub(q.x, p.x) : O_::sub(p.x, q.x);     // delta = p_a - p_b, a < b
                        T dy = (j < i) ? O_::sub(q.y, p.y) : O_::sub(p.y, q.y);
                        if (!(dx * dx + dy * dy >= c2_aa)) {                        // far pairs: see DESIGN.md cut-off
                            T fx, fy;
                            contact_force<T>(dx, dy, dmin_aa, a.margin, a.cforce, &fx, &fy);
                            if (j < i) { Fx = O_::add(-fx, Fx); Fy = O_::add(-fy, Fy); }
                            else       { Fx = O_::add(fx, Fx);  Fy = O_::add(fy, Fy); }
                        }
                    }
                    // agent (entity a) against every obstacle (entity b > a): force_a = (m_b / m_a) * force
                    const R2* envo = s_lm + le * L + LG;
                    const T ratio = O_::div(a.omass, a.mass);
                    for (int k = 0; k < NO; ++k) {
                        R2 q = envo[k];
                        T dx = O_::sub(p.x, q.x), dy = O_::sub(p.y, q.y);
                        if (!(dx * dx + dy * dy >= c2_ao)) {
                            T fx, fy;
                            contact_force<T>(dx, dy, dmin_ao, a.margin, a.cforce, &fx, &fy);
                            Fx = O_::add(O_::mul(ratio, fx), Fx); Fy = O_::add(O_::mul(ratio, fy), Fy);
                        }
                    }
                }
                for (int w = 0; w < a.n_walls; ++w) {                            // core.py:255-261
                    T fx, fy;
                    wall_force<T>(a.walls[w], p.x, p.y, a.size, a.margin, a.cforce, &fx, &fy);
                    Fx = O_::add(Fx, fx); Fy = O_::add(Fy, fy);
                }
                v.x = O_::mul(v.x, a.keep); v.y = O_::mul(v.y, a.keep);            // core.py:268
                v.x = O_::add(v.x, O_::mul(a.mass_one ? Fx : O_::div(Fx, a.mass), a.dt));
                v.y = O_::add(v.y, O_::mul(a.mass_one ? Fy : O_::div(Fy, a.mass), a.dt));
                if (a.has_vmax) {
                    T sp = O_::sqrt_(O_::sq2(v.x, v.y));
                    if (sp > a.vmax) { v.x = O_::mul(O_::div(v.x, sp), a.vmax); v.y = O_::mul(O_::div(v.y, sp), a.vmax); }
                }
                p.x = O_::add(p.x, O_::mul(v.x, a.dt));
                p.y = O_::add(p.y, O_::mul(v.y, a.dt));
                s_new[t] = p; s_v[t] = v;
                if (ts == a.n_steps - 1) { a.pos[g] = p; a.vel[g] = v; if (a.comm) a.comm[g] = O_::make((T)0, (T)0); }
            }
            // obstacles: one thread per (env, obstacle); contributions arrive in entity order -- agents
            // (obstacle is entity b: -(1/ratio) * force), earlier obstacles (b), later obstacles (a)
            for (int q = t; q < nvalid * NO; q += kBlock) {
                const int qe = q / NO, k = q - qe * NO;
                const R2* envo = s_lm + qe * L + LG;
                const R2 po = envo[k];
                T Fx = (T)0, Fy = (T)0;                                          // p_force[b] = 0.0 (core.py:252-253)
                const bool nf = env_nf(qe);
                const T c2_ao = env_cut2(cut2_ao, nf), c2_oo = env_cut2(cut2_oo, nf);
                if (a.collide) {
                    const R2* envp = s_old + qe * N;
                    const T c = -O_::div((T)1, O_::div(a.omass, a.mass));
                    for (int j = 0; j < N; ++j) {
                        R2 pj = envp[j];
                        T dx = O_::sub(pj.x, po.x), dy = O_::sub(pj.y, po.y);
                        if (!(dx * dx + dy * dy >= c2_ao)) {
                            T fx, fy;
                            contact_force<T>(dx, dy, dmin_ao, a.margin, a.cforce, &fx, &fy);
                            Fx = O_::add(O_::mul(c, fx), Fx); Fy = O_::add(O_::mul(c, fy), Fy);
                        }
                    }
                }
                for (int m = 0; m < NO; ++m) {
                    if (m == k) continue;
                    R2 q2 = envo[m];
                    T dx = (m < k) ? O_::sub(q2.x, po.x) : O_::sub(po.x, q2.x);
                    T dy = (m < k) ? O_::sub(q2.y, po.y) : O_::sub(po.y, q2.y);
                    if (!(dx * dx + dy * dy >= c2_oo)) {
                        T fx, fy;
                        contact_force<T>(dx, dy, dmin_oo, a.margin, a.cforce, &fx, &fy);
                        if (m < k) { Fx = O_::add(-fx, Fx); Fy = O_::add(-fy, Fy); }     // equal obstacle masses
                        else       { Fx = O_::add(fx, Fx);  Fy = O_::add(fy, Fy); }
                    }
                }
                for (int w = 0; w < a.n_walls; ++w) {
                    T fx, fy;
                    wall_force<T>(a.walls[w], po.x, po.y, a.osize, a.margin, a.cforce, &fx, &fy);
                    Fx = O_::add(Fx, fx); Fy = O_::add(Fy, fy);
                }
                R2 ov = s_ov[q];
                ov.x = O_::mul(ov.x, a.keep); ov.y = O_::mul(ov.y, a.keep);
                ov.x = O_::add(ov.x, O_::mul(O_::div(Fx, a.omass), a.dt));
                ov.y = O_::add(ov.y, O_::mul(O_::div(Fy, a.omass), a.dt));
                s_on[q] = O_::make(O_::add(po.x, O_::mul(ov.x, a.dt)), O_::add(po.y, O_::mul(ov.y, a.dt)));
                if (!OBSREW) {                                                   // World.step alone: write back and leave
                    const size_t gi = (size_t)(tile0 + qe) * L + LG + k;
                    a.lm[gi] = s_on[q];
                    if (a.lmv) a.lmv[gi] = ov;
                }
            }
            if (!OBSREW) { tick_arrive(a.tick_dev, gridDim.x, a.n_steps, t == 0); return; }
            __syncthreads();
        }

        // ================= Scenario.reward on the NEW state (formation_hd_obs_env.py:70-99) ======
        if (active && (!(fabs(p.x) < (T)INFINITY) || !(fabs(p.y) < (T)INFINITY))) s_bad[le] = 1;
        if (t < 2 * nvalid) {                                                    // np.mean(u, 0), np.mean(v, 0)
            const int qe = t >> 1;
            const int cnt = (t & 1) ? LG : N;
            const R2* src = (t & 1) ? (s_lm + qe * L) : (s_new + qe * N);
            T sx = 0, sy = 0;
            for (int j = 0; j < cnt; ++j) { R2 q = src[j]; sx = O_::add(sx, q.x); sy = O_::add(sy, q.y); }
            s_mean[t] = O_::make(O_::div(sx, (T)cnt), O_::div(sy, (T)cnt));
        }
        __syncthreads();
        if (active) {
            const R2 mp = s_mean[2 * le];
            s_cen[t] = O_::make(O_::sub(p.x, mp.x), O_::sub(p.y, mp.y));
        }
        __syncthreads();
        int col = 0;
        if (active) {
            if (a.collide) {                                                     // :91-97, is_collision :147-149
                const R2* envp = s_new + le * N;
                for (int j = 0; j < N; ++j) {
                    if (j == i) continue;
                    R2 q = envp[j];
                    if (O_::norm2(O_::sub(q.x, p.x), O_::sub(q.y, p.y)) < dmin_aa) ++col;
                }
                const R2* envo = s_on + le * NO;
                for (int k = 0; k < NO; ++k) {
                    R2 q = envo[k];
                    if (O_::norm2(O_::sub(q.x, p.x), O_::sub(q.y, p.y)) < dmin_ao) ++col;
                }
            }
            const R2 Ci = s_cen[t], ml = s_mean[2 * le + 1];                     // Hausdorff rows (:74-78)
            const R2* envl = s_lm + le * L;
            T rowmin = (T)INFINITY;
            for (int k = 0; k < LG; ++k) {
                R2 l = envl[k];
                rowmin = fmin(rowmin, O_::sq2(O_::sub(Ci.x, O_::sub(l.x, ml.x)), O_::sub(Ci.y, O_::sub(l.y, ml.y))));
            }
            atomicMax(&s_rowmax[le], O_::bits(rowmin));
            if (col) atomicAdd(&s_col[le], col);
        }
        for (int q = t; q < nvalid * LG; q += kBlock) {                          // Hausdorff columns
            const int qe = q / LG, k = q - qe * LG;
            const R2 ml = s_mean[2 * qe + 1];
            const R2 l = s_lm[qe * L + k];
            const R2 V = O_::make(O_::sub(l.x, ml.x), O_::sub(l.y, ml.y));
            const R2* envc = s_cen + qe * N;
            T colmin = (T)INFINITY;
            for (int j = 0; j < N; ++j) {
                R2 Cj = envc[j];
                colmin = fmin(colmin, O_::sq2(O_::sub(Cj.x, V.x), O_::sub(Cj.y, V.y)));
            }
            atomicMax(&s_rowmax[qe], O_::bits(colmin));
        }
        __syncthreads();

        stp += 1;                                                                // environment.py:114
        const bool dn = active && a.step && (stp >= a.world_length);
        if (active && i == 0) s_dn[le] = dn ? 1 : 0;
        if (active) {
            T base = -O_::sqrt_(O_::from_bits(s_rowmax[le]));
            if (s_bad[le]) base = O_::from_bits(~(Bits)0 >> 1);
            T r = base;
            for (int c = 0; c < col; ++c) r = O_::sub(r, (T)2);                   // rew -= 2 per collision
            const int coltot = s_col[le];
            const double R = (double)N * (double)base - 2.0 * (double)coltot;    // environment.py:136
            if (!FINOBS) a.reward[g] = (T)R;
            if (a.indiv) a.indiv[g] = r;
            if (a.done) a.done[g] = (uint8_t)(a.step ? (stp >= a.world_length) : 0);
            if (i == 0 && a.nan_flag && s_bad[le]) a.nan_flag[e] = 1;           // the reference's failure mode (Q9), sticky
            if (i == 0 && a.step) {
                T ret = (T)R;
                if (a.ep_return) { ret = a.ep_return[e] + (T)R; a.ep_return[e] = (dn && a.auto_reset) ? (T)0 : ret; }
                int ec = coltot;
                if (a.ep_coll) { ec += a.ep_coll[e]; a.ep_coll[e] = (dn && a.auto_reset) ? 0 : ec; }
                if (dn && a.stats) {
                    atomicAdd(&s_stat[0], 1.0);
                    atomicAdd(&s_stat[1], (double)ret);
                    atomicAdd(&s_stat[2], (double)ret * (double)ret);
                    atomicAdd(&s_stat[3], (double)ec);
                }
            }
        }
        // the reward hook's side effect (formation_hd_obs_env.py:85-88): obstacle velocities for the next step
        for (int q = t; q < nvalid * NO; q += kBlock)
            s_ov[q] = O_::make((T)0, (s_on[q].y > a.ofloor) ? a.ofall : (T)0);

        // ======== VecEnv auto-reset (env_wrappers.py:14-18; reset_world formation_hd_obs_env.py:101-120)
        if (PHYS && a.auto_reset) {
            if (__syncthreads_or(dn ? 1 : 0)) {
                const uint32_t tk = tick0 + (uint32_t)ts;
                if (dn) {
                    if (EXT && a.fin_pos) { a.fin_pos[g] = p; a.fin_vel[g] = v; }   // terminal block: post-step state
                    U4 r = philox(a.seed, ge, (uint32_t)i, tk, kResetAgent);
                    p = O_::make(uniform_pm1<T>(r.x), uniform_pm1<T>(r.y));
                    v = O_::make((T)0, (T)0);
                    s_new[t] = p; s_v[t] = v;
                    stp = 0;
                    if (ts == a.n_steps - 1) { a.pos[g] = p; a.vel[g] = v; }
                }
                for (int q = t; q < nvalid * L; q += kBlock) {
                    const int qe = q / L, k = q - qe * L;
                    if (!s_dn[qe]) continue;
                    if (EXT && a.fin_pos)                    // goals, then the obstacles at their post-step positions
                        a.fin_lm[(size_t)tile0 * L + q] = k < LG ? s_lm[q] : s_on[qe * NO + (k - LG)];
                    const uint32_t gq = a.env_offset + (uint32_t)(tile0 + qe);
                    if (k < LG) {
                        U4 r = philox(a.seed, gq, (uint32_t)k, tk, kResetLandmark);
                        s_lm[q] = O_::make(uniform_pm1<T>(r.x), uniform_pm1<T>(r.y));
                    } else {
                        R2 po, ov;
                        obstacle_reset<T>(a.seed, gq, k, k - LG, NO, tk, &po, &ov, a.ofall);
                        s_on[qe * NO + (k - LG)] = po; s_ov[qe * NO + (k - LG)] = ov;
                    }
                }
                __syncthreads();
            }
        }
        if (active && i == 0 && a.step) a.step[e] = stp;
        __syncthreads();                                                         // s_on / s_ov / s_lm final for this step

        // write back the landmarks (goals change only at a reset) and the obstacle velocities
        if (!PHYS || ts == a.n_steps - 1) {
            for (int q = t; q < nvalid * L; q += kBlock) {
                const int qe = q / L, k = q - qe * L;
                const size_t gi = (size_t)tile0 * L + q;
                if (k < LG) { if (PHYS && a.auto_reset) a.lm[gi] = s_lm[q]; }      // redrawn by an in-kernel reset
                else {
                    if (PHYS) a.lm[gi] = s_on[qe * NO + (k - LG)];
                    if (a.lmv) a.lmv[gi] = s_ov[qe * NO + (k - LG)];
                }
            }
        }

        // ================= observation rows (formation_hd_obs_env.py:53-68) =====================
        // [p_vel | goal landmarks (absolute) | obstacles - p_i | p_j - p_i (j != i) | comm zeros]
        if (a.obs && (!PHYS || ts == a.n_steps - 1)) {
            const int IPR = a.IPR;
            const uint32_t total = (uint32_t)(nvalid * N * IPR);
            R2* out = a.obs + (size_t)tile0 * N * IPR;
            for (uint32_t q = t; q < total; q += kBlock) {
                const uint32_t row = fastdiv(q, a.magic_ipr);
                const int k = (int)(q - row * IPR);
                const int rle = (int)fastdiv(row, a.magic_n);
                const int ri = (int)row - rle * N;
                R2 val;
                if (k == 0) val = s_v[row];
                else if (k < 1 + LG) val = s_lm[rle * L + (k - 1)];
                else if (k < 1 + LG + NO) {
                    const R2 o = s_on[rle * NO + (k - 1 - LG)], pi = s_new[row];
                    val = O_::make(O_::sub(o.x, pi.x), O_::sub(o.y, pi.y));
                } else if (k < 1 + LG + NO + (N - 1)) {
                    int j = k - (1 + LG + NO); j += (j >= ri);
                    const R2 pj = s_new[rle * N + j], pi = s_new[row];
                    val = O_::make(O_::sub(pj.x, pi.x), O_::sub(pj.y, pi.y));
                } else if (FINOBS && a.gth_rows) {
                    val = gather_record(a, tile0 + rle) < 0 ? nan2 : O_::make((T)0, (T)0);   // comm zeros; NaN slot
                } else val = O_::make((T)0, (T)0);
                out[q] = val;
            }
        }
        if (!PHYS) break;
        // next step of an in-kernel rollout: new state becomes the old one
        __syncthreads();
        R2* tmp = s_old; s_old = s_new; s_new = tmp;
        for (int q = t; q < nvalid * NO; q += kBlock) {
            const int qe = q / NO, k = q - qe * NO;
            s_lm[qe * L + LG + k] = s_on[q];
        }
    }
    if (a.stats) {
        __syncthreads();
        if (t < 4 && s_stat[0] != 0.0) atomicAdd(&a.stats[t], s_stat[t]);
    }
    if (PHYS) tick_arrive(a.tick_dev, gridDim.x, a.n_steps, t == 0);
}

// Scenario.reset_world (formation_hd_obs_env.py:101-120) for masked envs; same Philox counters as the in-kernel
// auto-reset.
template <typename T>
__global__ void k_reset_obst(const __grid_constant__ KArgs<T> a, const uint8_t* __restrict__ mask) {
    typedef Ops<T> O_;
    typedef typename O_::R2 R2;
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= a.E) return;
    if (mask && !mask[e]) return;
    const int N = a.N, L = a.L, NO = a.n_obst, LG = a.L - a.n_obst;
    const uint32_t ge = a.env_offset + (uint32_t)e;
    const uint32_t tick0 = a.tick + (a.tick_dev ? a.tick_dev[0] : 0u);
    const R2 zero = O_::make((T)0, (T)0);
    for (int i = 0; i < N; ++i) {
        U4 r = philox(a.seed, ge, (uint32_t)i, tick0, kResetAgent);
        const size_t g = (size_t)e * N + i;
        a.pos[g] = O_::make(uniform_pm1<T>(r.x), uniform_pm1<T>(r.y));
        a.vel[g] = zero;
        if (a.comm) a.comm[g] = zero;
    }
    for (int k = 0; k < L; ++k) {
        const size_t gi = (size_t)e * L + k;
        if (k < LG) {
            U4 r = philox(a.seed, ge, (uint32_t)k, tick0, kResetLandmark);
            a.lm[gi] = O_::make(uniform_pm1<T>(r.x), uniform_pm1<T>(r.y));
            if (a.lmv) a.lmv[gi] = zero;
        } else {
            R2 po, ov;
            obstacle_reset<T>(a.seed, ge, k, k - LG, NO, tick0, &po, &ov, a.ofall);
            a.lm[gi] = po;
            if (a.lmv) a.lmv[gi] = ov;
        }
    }
    if (a.step) a.step[e] = 0;
    if (a.ep_return) a.ep_return[e] = (T)0;
    if (a.ep_coll) a.ep_coll[e] = 0;
}

}  // namespace fg
