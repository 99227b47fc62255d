#pragma once
// fg_abi_impl.cuh -- implementation of the extern "C" entry points declared in include/formation_gym_b200.h,
// templated on the real type; fg_abi_f32.cu / fg_abi_f64.cu instantiate one precision each (two translation units,
// compiled in parallel by formation_gym/_build.py).
// Validates arguments, converts fg_params (double) into the kernels' typed argument block and
// launches asynchronously on the caller's stream.  No allocation, no global state, no sync.
#include <cstring>
#include <cmath>
#include <cstdlib>
#include <type_traits>
#include <algorithm>

#include "fg_host.cuh"
#include "fg_kernels.cuh"
#include "fg_warp.cuh"
#include "fg_obstacle.cuh"
#include "fg_policy.cuh"

namespace fgabi {
// warp-autonomous kernel of the partial-observation scenarios (fg_lm_f32.cu / fg_lm_f64.cu): FG_OK / error code, or 1
// when there is no instantiation for this (scenario, N, L, num_obs)
int launch_lm_warp(const fg::KArgs<float>& a, int scenario, cudaStream_t st);
int launch_lm_warp(const fg::KArgs<double>& a, int scenario, cudaStream_t st);
}  // namespace fgabi

namespace {

uint32_t magic_for(int d) {          // floor(2^32 / d) + 1; 0 encodes d == 1 (fastdiv returns q)
    if (d <= 1) return 0u;
    return (uint32_t)((((uint64_t)1) << 32) / (uint64_t)d) + 1u;
}

template <typename T> double kcut_for();
// Contact cut-off in units of contact_margin k: beyond d_min + kcut*k the softplus penetration is
// < k*exp(-kcut), i.e. the dropped force is < contact_force*k*exp(-kcut) = 0.1*exp(-kcut):
// fp32 build kcut = 20 -> 2e-10 (velocity error 2e-11, far below fp32 rounding of v and the 1e-5
// tolerance); fp64 build kcut = 50 -> 2e-23 (tolerance 1e-9 over 25 steps).
template <> double kcut_for<float>() { return 20.0; }
template <> double kcut_for<double>() { return 50.0; }

template <typename T>
int fill_args(fg::KArgs<T>& a, const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L,
              uint64_t seed, uint32_t tick, uint32_t env_offset) {
    typedef typename fg::Ops<T>::R2 R2;
    if (!p || !b) return fail(FG_ERR_ARG, "null params/buffers%s");
    if (E < 1) return fail(FG_ERR_ARG, "E must be >= 1%s");
    if (N < 1 || N > FG_MAX_AGENTS) return fail(FG_ERR_ARG, "N must be in [1, FG_MAX_AGENTS=256]%s");
    if (scenario == FG_SCENARIO_HD) {
        if (N < 3) return fail(FG_ERR_ARG, "formation_hd_env needs N >= 3 (formation_hd_env.py:58)%s");
        L = N;
    } else if (scenario == FG_SCENARIO_BASIC || scenario == FG_SCENARIO_HD_PARTIAL ||
               scenario == FG_SCENARIO_HD_PARTIAL_RANGE) {
        if (L < 1 || L > FG_MAX_LANDMARKS) return fail(FG_ERR_ARG, "L must be in [1, FG_MAX_LANDMARKS]%s");
        if (scenario == FG_SCENARIO_HD_PARTIAL && (p->num_obs < 0 || p->num_obs > 4 * FG_MAX_AGENTS))
            return fail(FG_ERR_ARG, "num_obs out of range%s");
    } else if (scenario == FG_SCENARIO_HD_OBSTACLE) {
        if (L < 1 || L > FG_MAX_LANDMARKS) return fail(FG_ERR_ARG, "L must be in [1, FG_MAX_LANDMARKS]%s");
        if (p->num_obstacles < 0 || p->num_obstacles >= L)
            return fail(FG_ERR_ARG, "num_obstacles must be in [0, L): L counts goal landmarks + obstacles%s");
        if (!p->silent) return fail(FG_ERR_ARG, "formation_hd_obs_env: silent agents only (formation_hd_obs_env.py:28)%s");
        if (p->agent_mass || p->agent_size_arr || p->agent_accel || p->agent_max_speed)
            return fail(FG_ERR_ARG, "formation_hd_obs_env: per-agent mass/size/accel/max_speed arrays are not supported%s");
        if (!(p->obstacle_size > 0.0) || !(p->obstacle_mass > 0.0))
            return fail(FG_ERR_ARG, "formation_hd_obs_env: obstacle_size and obstacle_mass must be positive%s");
    } else {
        return fail(FG_ERR_ARG, "unknown scenario id%s");
    }
    if ((uint64_t)E * (uint64_t)N >= (1ull << 31)) return fail(FG_ERR_ARG, "E*N must be < 2^31%s");
    if (p->n_walls < 0 || p->n_walls > FG_MAX_WALLS) return fail(FG_ERR_ARG, "n_walls out of range%s");
    {
        // every 2-vector buffer is accessed as float2 / double2 items
        const void* vec[] = {b->pos, b->vel, b->act, b->comm, b->ideal_shape, b->ideal_vel, b->landmarks,
                             b->landmark_vel, b->obs};
        for (const void* q : vec)
            if (q && ((uintptr_t)q % sizeof(R2)) != 0)
                return fail(FG_ERR_ARG, "2-vector buffers (pos, vel, act, comm, ideal_*, landmarks, obs) must be "
                                        "8-byte (fp32) / 16-byte (fp64) aligned%s");
    }
    memset(&a, 0, sizeof(a));
    a.pos = (R2*)b->pos; a.vel = (R2*)b->vel; a.act = (const R2*)b->act; a.comm = (R2*)b->comm;
    a.shape = (R2*)b->ideal_shape; a.ivel = (R2*)b->ideal_vel; a.lm = (R2*)b->landmarks;
    a.step = b->step; a.obs = (R2*)b->obs; a.reward = (T*)b->reward; a.indiv = (T*)b->indiv;
    a.done = b->done; a.ep_return = (T*)b->ep_return; a.ep_coll = b->ep_collisions; a.stats = b->stats;
    a.tick_dev = b->tick_dev; a.nan_flag = b->nan_flag; a.cpos = (const R2*)b->contact_pos;
    a.a_mass = (const T*)p->agent_mass; a.a_size = (const T*)p->agent_size_arr;
    a.a_accel = (const T*)p->agent_accel; a.a_vmax = (const T*)p->agent_max_speed;
    a.E = E; a.N = N; a.L = L;
    a.EPC = fg::kBlock / N;
    a.IPR = scenario == FG_SCENARIO_HD ? 3 * N
          : scenario == FG_SCENARIO_BASIC ? 2 + L + 2 * (N - 1)
          : scenario == FG_SCENARIO_HD_PARTIAL ? 1 + L + p->num_obs + (N - 1)
          : 1 + L + 2 * (N - 1);                    // partial range; obstacle: 1 + goals + obstacles + 2(N-1)
    a.lmv = (R2*)b->landmark_vel; a.n_obst = scenario == FG_SCENARIO_HD_OBSTACLE ? p->num_obstacles : 0;
    a.osize = (T)p->obstacle_size; a.omass = (T)p->obstacle_mass;
    a.ofloor = (T)p->obstacle_floor; a.ofall = (T)p->obstacle_fall_vy;
    a.num_obs = p->num_obs; a.obs_range = (T)p->obs_range;
    a.magic_n = magic_for(N); a.magic_ipr = magic_for(a.IPR);
    a.magic_l = magic_for(L); a.magic_np = magic_for((N + 31) & ~31);
    a.act_r2 = p->silent ? 1 : 2;
    a.dt = (T)p->dt; a.keep = (T)(1.0 - p->damping); a.cforce = (T)p->contact_force;
    a.margin = (T)p->contact_margin; a.size = (T)p->agent_size; a.mass = (T)p->mass;
    a.vmax = (T)p->max_speed; a.u_noise = (T)p->u_noise; a.c_noise = (T)p->c_noise;
    a.sens0 = (T)p->sensitivity; a.accel = (T)p->accel;
    a.has_accel = p->has_accel; a.has_vmax = p->has_max_speed;
    a.sens = p->action_prescaled ? (T)1 : (p->has_accel ? (T)p->accel : (T)p->sensitivity);
    a.prescaled = p->action_prescaled;
    a.gain = p->has_accel ? (T)((T)p->mass * (T)p->accel) : (T)p->mass;
    a.mass_one = (p->mass == 1.0);
    a.kcut = (T)kcut_for<T>();
    {
        T dmin = a.size + a.size;
        T c = dmin + a.kcut * a.margin;
        a.cut2 = c * c;
        // hd: (s1+s2)/2 (formation_hd_env.py:121); basic: s1+s2 (basic_formation_env.py:91)
        a.rthr = scenario == FG_SCENARIO_HD ? dmin / (T)2 : dmin;
        a.rthr2_hi = a.rthr * a.rthr * (T)1.0001;
    }
    a.collide = p->collide; a.silent = p->silent; a.world_length = p->world_length;
    a.n_walls = p->n_walls;
    for (int w = 0; w < p->n_walls; ++w) {
        a.walls[w].orient = p->walls[w].orient; a.walls[w].hard = p->walls[w].hard;
        a.walls[w].axis_pos = (T)p->walls[w].axis_pos; a.walls[w].end0 = (T)p->walls[w].end0;
        a.walls[w].end1 = (T)p->walls[w].end1; a.walls[w].width = (T)p->walls[w].width;
    }
    a.n_steps = 1; a.random_actions = 0; a.auto_reset = 0;
    {
        // warp kernel: L2 prefetch of the state two spans ahead (fg_warp.cuh) once the four per-agent state arrays
        // (pos, vel, act, ideal_shape) no longer stay resident in the 126 MB L2 next to the observation stream.
        // Measured (B200, fp32, step kernel alone): N = 27 x 65536 envs (57 MB of state) 0.80 -> 0.90 of the HBM peak,
        // N = 27 x 262144 0.72 -> 0.87, basic N = 3 x 1 M 0.66 -> 0.72; but N = 9 x 131072 (38 MB, L2-resident)
        // 0.95 -> 0.88: each prefetch.global.L2 holds its warp for an L2 round trip.
        const int mode = fgabi::switches().l2_prefetch.load(std::memory_order_relaxed);       // 0 never, 1 auto, 2 always
        const double state_bytes = (double)E * (double)N * 4.0 * (double)sizeof(R2);
        a.pf_dist = mode == 2 || (mode == 1 && state_bytes > 44e6) ? fgabi::switches().pf_spans.load(std::memory_order_relaxed) : 0;
    }
    a.seed = seed; a.tick = tick; a.env_offset = env_offset;
    // long hd rows of silent agents: static 2/3 of each row bulk-stored from one shared image
    // (measured: N = 243 270 us vs 353 us with plain stores; break-even near N = 50)
    {
        const fgabi::Switches& sw = fgabi::switches();                 // A/B switches for tests and profiling
        // measured (scripts/quick_cfg.py): without observations the packed loops win from N = 32 up (N = 243:
        // 93 -> 59 us per 1024 envs); with observations the kernel is bound by its obs writer and the extra
        // shared memory only pays for large N
        a.fast_pairs = N >= 32 && (!b->obs || N >= 64 || sw.force_fast_pairs.load(std::memory_order_relaxed)) &&
                       !sw.no_fast_pairs.load(std::memory_order_relaxed) && !b->contact_pos;
    }
    {
        // hashed cell lists of the packed pair loops (fg_pairs.cuh): buckets per env = largest power of two
        // <= 4 * roundup(N, 32); cell edge = 2 * search radius * (1 + 2^-9)
        const int NP = (N + 31) & ~31;
        int logb = 0;
        while ((2 << logb) <= 4 * NP) ++logb;
        a.cell_shift = 32 - logb;
        a.cells = a.fast_pairs && p->collide && !fgabi::switches().no_cells.load(std::memory_order_relaxed);
        a.cell_inv_old = (float)(1.0 / (2.0 * std::sqrt((double)a.cut2) * (1.0 + 1.0 / 512.0)));
        a.cell_inv_new = (float)(1.0 / (2.0 * std::sqrt((double)a.rthr2_hi) * (1.0 + 1.0 / 512.0)));
        a.cell_off = 0;
    }
    a.row_tma = scenario == FG_SCENARIO_HD && p->silent && b->obs && ((uintptr_t)b->obs % sizeof(R2)) == 0 &&
                N >= fgabi::switches().row_min_n.load(std::memory_order_relaxed);
    a.row_nbuf = fgabi::switches().row_nbuf.load(std::memory_order_relaxed) == 1 ? 1 : 2;
    // chunked row writer (fg_kernels.cuh rows_chunked): the largest power-of-two row count <= 16 whose image fits 32 KB
    // Measured (B200, fp32, step kernel alone, chunked vs the round-1 writers): N = 10 0.57 vs 0.45 of the HBM peak (tile
    // image), 12 0.58 vs 0.34, 20 0.70 vs 0.29, 30 0.72 vs 0.40, 40 0.80 vs 0.42 (warp-per-row plain stores), 48 0.76 vs
    // 0.51, 56 0.77 vs 0.57, 63 0.82 vs 0.66, 64 0.74 vs 0.65, 72 0.73 vs 0.66 (per-row pieces), 75 / 81 equal, 100 0.82 vs
    // 0.84, 128 0.85 vs 0.88, 243 0.79 vs 0.89 (the single image stalls the CTA while its 23 KB chunk is read):
    // chunks for 10 <= N <= 80 (row_chunks = 2 forces them for every N >= row_min_n).
    a.row_chunk = 0; a.row_chunk_log2 = 0;
    const int rc_mode = fgabi::switches().row_chunks.load(std::memory_order_relaxed);
    if (a.row_tma && (rc_mode == 2 || (rc_mode == 1 && N <= 80))) {
        int lg = fgabi::switches().row_chunk_max_log2.load(std::memory_order_relaxed);
        while (lg > 1 && ((size_t)(1 << lg) * a.IPR + 2) * sizeof(R2) > 32 * 1024) --lg;
        if (((size_t)(1 << lg) * a.IPR + 2) * sizeof(R2) <= 48 * 1024) { a.row_chunk = 1 << lg; a.row_chunk_log2 = lg; }
    }
    a.row_early = a.row_tma && sizeof(R2) == 8 && (a.row_chunk || ((N & 1) && ((uintptr_t)b->obs % 16) == 0)) &&
                  !fgabi::switches().no_early_rows.load(std::memory_order_relaxed);
    return FG_OK;
}

// Target bank (fg_targets): validated before anything else (no device call on a bad argument); tg == NULL = no bank.
template <typename T>
int check_targets(const fg_targets* tg, int scenario, const char* who) {
    typedef typename fg::Ops<T>::R2 R2;
    if (!tg) return FG_OK;
    if (scenario != FG_SCENARIO_HD)
        return fail(FG_ERR_ARG, "%s: target banks are defined for formation_hd_env only", who);
    if (tg->count < 1) return fail(FG_ERR_ARG, "%s: fg_targets.count must be >= 1", who);
    if (!tg->shapes) return fail(FG_ERR_ARG, "%s: fg_targets.shapes must be non-null", who);
    if (((uintptr_t)tg->shapes % sizeof(R2)) != 0 || ((uintptr_t)tg->vels % sizeof(R2)) != 0)
        return fail(FG_ERR_ARG, "%s: fg_targets.shapes / vels must be 8-byte (fp32) / 16-byte (fp64) aligned", who);
    if (((uintptr_t)tg->index % sizeof(int32_t)) != 0)
        return fail(FG_ERR_ARG, "%s: fg_targets.index must be 4-byte aligned", who);
    return FG_OK;
}

template <typename T>
void set_targets(fg::KArgs<T>& a, const fg_targets* tg) {
    typedef typename fg::Ops<T>::R2 R2;
    if (!tg) return;                                                // fill_args left the bank empty (count 0)
    a.tgt_shape = (const R2*)tg->shapes; a.tgt_vel = (const R2*)tg->vels;
    a.tgt_index = tg->index; a.tgt_count = tg->count;
}

// Terminal block (fg_final): validated before anything else (no device call on a bad argument); f == NULL = no block.
// step != 0: a step entry point (auto-reset on, one step per call: then the mask of written envs is the step's done).
template <typename T>
int check_final(const fg_final* f, const fg_params* p, int scenario, int auto_reset, int n_steps, bool step,
                const char* who) {
    typedef typename fg::Ops<T>::R2 R2;
    if (!f) return FG_OK;
    if (step && !auto_reset) return fail(FG_ERR_ARG, "%s: a terminal block needs auto_reset != 0", who);
    if (step && n_steps != 1) return fail(FG_ERR_ARG, "%s: a terminal block needs n_steps == 1", who);
    if (!f->pos || !f->vel) return fail(FG_ERR_ARG, "%s: fg_final.pos / vel must be non-null", who);
    if (scenario == FG_SCENARIO_HD && (!f->ideal_shape || !f->ideal_vel))
        return fail(FG_ERR_ARG, "%s: fg_final.ideal_shape / ideal_vel must be non-null for formation_hd_env", who);
    if (scenario != FG_SCENARIO_HD && !f->landmarks)
        return fail(FG_ERR_ARG, "%s: fg_final.landmarks must be non-null for this scenario", who);
    if (p && !p->silent && !f->comm) return fail(FG_ERR_ARG, "%s: fg_final.comm must be non-null for non-silent agents", who);
    const void* vec[] = {f->pos, f->vel, f->comm, f->ideal_shape, f->ideal_vel, f->landmarks};
    for (const void* q : vec)
        if (((uintptr_t)q % sizeof(R2)) != 0)
            return fail(FG_ERR_ARG, "%s: fg_final arrays must be 8-byte (fp32) / 16-byte (fp64) aligned", who);
    return FG_OK;
}

template <typename T>
void set_final(fg::KArgs<T>& a, const fg_final* f, const fg_params* p, int scenario) {
    typedef typename fg::Ops<T>::R2 R2;
    if (!f) return;                                                 // fill_args left the block empty (fin_pos NULL)
    a.fin_pos = (R2*)f->pos; a.fin_vel = (R2*)f->vel;
    a.fin_comm = p->silent ? nullptr : (R2*)f->comm;
    if (scenario == FG_SCENARIO_HD) { a.fin_shape = (R2*)f->ideal_shape; a.fin_ivel = (R2*)f->ideal_vel; }
    else a.fin_lm = (R2*)f->landmarks;
}

template <typename T>
size_t smem_bytes(const fg::KArgs<T>& a, int scenario, bool het) {
    typedef typename fg::Ops<T>::R2 R2;
    typedef typename fg::Ops<T>::Bits Bits;
    const size_t nA = (size_t)a.EPC * a.N;
    const size_t nS = scenario == FG_SCENARIO_HD ? nA : (size_t)a.EPC * a.L;
    size_t s = (4 * nA + nS + 3 * a.EPC + (scenario != FG_SCENARIO_BASIC ? nA : 0)) * sizeof(R2)
               + a.EPC * sizeof(Bits);
    if (scenario == FG_SCENARIO_BASIC) s += (size_t)a.EPC * a.L * sizeof(T);
    if (het) s += 5 * (size_t)a.N * sizeof(T);
    s += 3 * a.EPC * sizeof(int);
    if (a.row_tma && a.row_chunk)                                       // one image of row_chunk rows (+ phase slack)
        s += (size_t)(((size_t)a.row_chunk * a.IPR + 3) & ~(size_t)1) * sizeof(R2);
    else if (a.row_tma)                                                 // static row images + per-warp staging
        s += ((size_t)2 * (2 * a.N + 1) * a.EPC + (size_t)a.row_nbuf * ((a.N + 3) & ~1) * (fg::kBlock / 32)) * sizeof(R2);
    return (s + 15) & ~(size_t)15;
}

// OM == 3 (short rows staged per thread, one bulk store per tile): image of EPC*N rows (+ phase items)
template <typename T>
size_t tile_image_bytes(const fg::KArgs<T>& a) {
    typedef typename fg::Ops<T>::R2 R2;
    return (size_t)(((size_t)a.EPC * a.N * a.IPR + 3) & ~(size_t)1) * sizeof(R2);
}
template <typename T>
bool tile_image_ok(const fg::KArgs<T>& a) {
    typedef typename fg::Ops<T>::R2 R2;
    return a.obs && ((uintptr_t)a.obs % sizeof(R2)) == 0 && tile_image_bytes(a) <= 96 * 1024 &&
           !fgabi::switches().no_tile_image.load(std::memory_order_relaxed);
}

// extra shared memory of the fast pair loops: 8 arrays of EPC*roundup(N,32) floats, the per-(env,warp)
// partial sums and the two max-norm words per env
template <typename T>
size_t fast_pairs_bytes(const fg::KArgs<T>& a) {
    const size_t NP = ((size_t)a.N + 31) & ~(size_t)31;
    return (8 * (size_t)a.EPC * NP + (size_t)a.EPC * 32) * sizeof(float) + 2 * (size_t)a.EPC * sizeof(unsigned) + 16;
}

// Tile kernels (k_step, k_step_obst): EPC envs per CTA of kBlock threads
template <auto Kernel, typename T>
int launch_tile(const fg::KArgs<T>& a, size_t smem, cudaStream_t st) {
    cudaError_t err = ensure_dyn_smem<Kernel>(smem);
    if (err != cudaSuccess) return fail(FG_ERR_CUDA, "cudaFuncSetAttribute failed: %s", cudaGetErrorString(err));
    Kernel<<<(a.E + a.EPC - 1) / a.EPC, fg::kBlock, smem, st>>>(a);
    return launch_status();
}

template <typename T, int SCN, bool PHYS, bool OBSREW, bool HET, int OM, bool FP, bool EXT>
int launch_one_ext(const fg::KArgs<T>& a, size_t smem, cudaStream_t st) {
    fg::KArgs<T> b = a;
    if (FP) {
        smem += fast_pairs_bytes(a);
        if (a.cells) {                      // chain nodes [2][EPC][NP] x 16 B, bucket heads [2][EPC][CB], flags [2][EPC]
            smem = (smem + 15) & ~(size_t)15;
            b.cell_off = (unsigned)smem;
            const size_t NP = ((size_t)a.N + 31) & ~(size_t)31, CB = (size_t)1 << (32 - a.cell_shift);
            smem += 2 * (size_t)a.EPC * CB * sizeof(int) + 2 * (size_t)a.EPC * NP * 16 + 2 * (size_t)a.EPC * sizeof(int);
            smem = (smem + 15) & ~(size_t)15;
        }
    } else {
        b.cells = 0;
    }
    return launch_tile<fg::k_step<T, SCN, PHYS, OBSREW, HET, OM, FP, EXT>>(b, smem, st);
}

// steps with a target bank or a terminal block, and fg_final_obs, take the EXT instantiation of the same kernel
template <typename T, int SCN, bool PHYS, bool OBSREW, bool HET, int OM, bool FP>
int launch_one(const fg::KArgs<T>& a, size_t smem, cudaStream_t st) {
    if constexpr (OBSREW)
        if (fg::reset_ext(a)) return launch_one_ext<T, SCN, PHYS, OBSREW, HET, OM, FP, true>(a, smem, st);
    return launch_one_ext<T, SCN, PHYS, OBSREW, HET, OM, FP, false>(a, smem, st);
}

// Fast pair loops (fg_pairs.cuh): fp32, formation_hd_env, uniform agents, 32 <= N (a warp spans <= 2 envs).
template <typename T, int SCN, bool PHYS, bool OBSREW, bool HET, int OM>
int launch_fp(const fg::KArgs<T>& a, size_t smem, cudaStream_t st) {
    constexpr bool kCan = std::is_same<T, float>::value && SCN == fg::kScnHD && !HET;
    if (kCan && a.fast_pairs) return launch_one<T, SCN, PHYS, OBSREW, HET, OM, kCan>(a, smem, st);
    return launch_one<T, SCN, PHYS, OBSREW, HET, OM, false>(a, smem, st);
}

// observation-writer mode of the tile kernel (fg_kernels.cuh k_step<..., OM>)
template <typename T, int SCN, bool PHYS, bool OBSREW, bool HET>
int launch_om(const fg::KArgs<T>& a, size_t smem, cudaStream_t st) {
    if (!OBSREW) return launch_fp<T, SCN, PHYS, OBSREW, HET, 0>(a, smem, st);
    if (SCN == fg::kScnHD && a.row_tma) return launch_fp<T, SCN, PHYS, OBSREW, HET, (SCN == fg::kScnHD ? 2 : 0)>(a, smem, st);
    if (SCN < fg::kScnPartial && a.IPR >= 48) return launch_fp<T, SCN, PHYS, OBSREW, HET, 1>(a, smem, st);
    if (tile_image_ok<T>(a)) return launch_fp<T, SCN, PHYS, OBSREW, HET, (OBSREW ? 3 : 0)>(a, smem + tile_image_bytes<T>(a), st);
    return launch_fp<T, SCN, PHYS, OBSREW, HET, 0>(a, smem, st);
}

template <typename T, int SCN, bool PHYS, bool OBSREW>
int launch_het(const fg::KArgs<T>& a, bool het, size_t smem, cudaStream_t st) {
    return het ? launch_om<T, SCN, PHYS, OBSREW, true>(a, smem, st) : launch_om<T, SCN, PHYS, OBSREW, false>(a, smem, st);
}

template <typename T, bool PHYS, bool OBSREW>
int launch(const fg::KArgs<T>& a, int scenario, const fg_params* p, void* stream) {
    const bool het = p->agent_mass || p->agent_size_arr || p->agent_accel || p->agent_max_speed;
    const size_t smem = smem_bytes<T>(a, scenario, het);
    cudaStream_t st = (cudaStream_t)stream;
    if (scenario == FG_SCENARIO_HD) return launch_het<T, fg::kScnHD, PHYS, OBSREW>(a, het, smem, st);
    if (OBSREW && scenario == FG_SCENARIO_HD_PARTIAL) return launch_het<T, fg::kScnPartial, PHYS, OBSREW>(a, het, smem, st);
    if (OBSREW && scenario == FG_SCENARIO_HD_PARTIAL_RANGE) return launch_het<T, fg::kScnRange, PHYS, OBSREW>(a, het, smem, st);
    return launch_het<T, fg::kScnBasic, PHYS, OBSREW>(a, het, smem, st);
}


// formation_hd_obs_env (fg_obstacle.cuh)
template <typename T, bool PHYS, bool OBSREW, bool EXT>
int launch_obstacle_ext(const fg::KArgs<T>& a, void* stream) {
    typedef typename fg::Ops<T>::R2 R2;
    typedef typename fg::Ops<T>::Bits Bits;
    const size_t nA = (size_t)a.EPC * a.N;
    size_t smem = (4 * nA + (size_t)a.EPC * a.L + 2 * (size_t)a.EPC * a.n_obst + 2 * a.EPC) * sizeof(R2)
                  + a.EPC * sizeof(Bits) + 3 * a.EPC * sizeof(int);
    smem = (smem + 15) & ~(size_t)15;
    return launch_tile<fg::k_step_obst<T, PHYS, OBSREW, EXT>>(a, smem, (cudaStream_t)stream);
}

template <typename T, bool PHYS, bool OBSREW = true>
int launch_obstacle(const fg::KArgs<T>& a, void* stream) {
    if constexpr (OBSREW)
        if (fg::reset_ext(a)) return launch_obstacle_ext<T, PHYS, OBSREW, true>(a, stream);
    return launch_obstacle_ext<T, PHYS, OBSREW, false>(a, stream);
}

// ---- warp-autonomous kernels (fg_warp.cuh k_hd_warp, fg_warp_lm.cuh k_lm_warp) ---------------------
// Resident CTAs per SM for w warps per CTA (occupancy API; shared memory is the limiter: one
// observation-span image per warp).  Computed once per instantiation; all GPUs of a box are alike.
// LY: the kernel's layout (stride bytes of shared memory per warp, at most MAXW warps per CTA, EPW envs per span).
struct WarpGeom { int ctas[4]; int best; int sms; };      // index: log2(w), w = 1, 2, 4, 8

template <auto Kernel, typename LY>
const WarpGeom& warp_geom() {
    static const WarpGeom geom = [] {
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
            if (cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
                cudaGetLastError();
                continue;
            }
            int ctas = 0;
            if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas, Kernel, 32 * w, smem) != cudaSuccess) {
                cudaGetLastError();
                continue;
            }
            g_.ctas[l] = ctas;
            if (ctas * w > best_res) { best_res = ctas * w; g_.best = l; }
        }
        // the probing above left the limit at the SMALLEST footprint, and a limit below the launch's request makes
        // the launch fail (also under the 48 KB default): restore the default-or-larger value; launches raise it
        // further through ensure_dyn_smem when they need more than 48 KB
        cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 48 * 1024);
        cudaGetLastError();
        return g_;
    }();
    return geom;
}

// name: the kernel's name in the "does not fit" message
template <auto Kernel, typename LY, typename T>
int launch_persistent(const fg::KArgs<T>& a, const char* name, cudaStream_t st) {
    const WarpGeom& gm = warp_geom<Kernel, LY>();
    const int spans = (a.E + LY::EPW - 1) / LY::EPW;
    int l = gm.best;
    while (l > 0 && (spans >> l) < 2 * gm.sms) --l;                // small batches: spread over the SMs
    if (gm.ctas[l] < 1) return fail(FG_ERR_CUDA, "%s does not fit on this device", name);
    const int w = 1 << l;
    const size_t smem = (size_t)w * LY::stride;
    cudaError_t err = ensure_dyn_smem<Kernel>(smem);
    if (err != cudaSuccess) return fail(FG_ERR_CUDA, "cudaFuncSetAttribute failed: %s", cudaGetErrorString(err));
    // persistent warps: at most one resident wave; each warp walks spans gw, gw + nwarps, ...
    int grid = (spans + w - 1) / w;
    int wave = gm.sms * gm.ctas[l];
    wave *= std::max(1, fgabi::switches().waves.load(std::memory_order_relaxed));
    if (grid > wave) grid = wave;
    if ((grid * w) & 1) ++grid;                                    // even warp count (16-byte phase, fg_warp.cuh)
    Kernel<<<grid, 32 * w, smem, st>>>(a);
    return launch_status();
}

template <typename T, int N, bool WOBS, int SCN, bool STD, int POL = 0, bool EXT = false>
int launch_warp_ext(const fg::KArgs<T>& a, cudaStream_t st) {
    return launch_persistent<fg::k_hd_warp<T, N, WOBS, SCN, STD, POL, EXT>, fg::WarpLayout<T, N, WOBS>>(a, "k_hd_warp", st);
}

// runs with a target bank or a terminal block take the EXT instantiation of the same kernel
template <typename T, int N, bool WOBS, int SCN, bool STD, int POL = 0>
int launch_warp_n(const fg::KArgs<T>& a, cudaStream_t st) {
    if (fg::reset_ext(a)) return launch_warp_ext<T, N, WOBS, SCN, STD, POL, true>(a, st);
    return launch_warp_ext<T, N, WOBS, SCN, STD, POL, false>(a, st);
}

// The standard product configuration: the fp32 warp kernels have an STD instantiation with these run-time tests
// compiled out (fg_warp.cuh, fg_warp_lm.cuh).  Each caller decides what fp64 runs.
template <typename T>
bool std_config(const fg::KArgs<T>& a) {
    return a.collide && !a.has_vmax && a.mass_one && a.n_steps == 1 && a.step && a.done && a.indiv && a.ep_return &&
           a.ep_coll && a.stats && !a.comm && !fgabi::switches().no_std_kernel.load(std::memory_order_relaxed);
}

template <typename T, int N, int SCN = fg::kScnHD>
int launch_warp(const fg::KArgs<T>& a, cudaStream_t st) {
    // fp32 standard configuration: the STD instantiation; anything else (fp64 too) the generic one
    if constexpr (std::is_same<T, float>::value)
        if (std_config(a))
            return a.obs ? launch_warp_n<T, N, true, SCN, true>(a, st) : launch_warp_n<T, N, false, SCN, true>(a, st);
    return a.obs ? launch_warp_n<T, N, true, SCN, false>(a, st) : launch_warp_n<T, N, false, SCN, false>(a, st);
}

// What neither warp-autonomous kernel handles: per-agent constants, walls, non-silent agents, cached contact
// positions, unaligned observations; and the A/B switch for tests and profiling.
template <typename T>
bool warp_common_ok(const fg_params* p, const fg_buffers* b) {
    if (p->agent_mass || p->agent_size_arr || p->agent_accel || p->agent_max_speed) return false;
    if (p->n_walls != 0 || !p->silent || b->contact_pos) return false;
    if (((uintptr_t)b->obs) % sizeof(typename fg::Ops<T>::R2)) return false;
    return !fgabi::switches().force_tile_kernel.load(std::memory_order_relaxed);
}

// The fast path covers the configurations BASELINE.json names for formation_hd_env with N <= 27.
template <typename T>
bool warp_path_ok(const fg::KArgs<T>& a, int scenario, const fg_params* p, const fg_buffers* b) {
    if (scenario == FG_SCENARIO_BASIC) {
        if (a.N != 3 || a.L != a.N || !b->landmarks) return false;  // the default 3 agents / 3 landmarks
    } else {
        if (scenario != FG_SCENARIO_HD) return false;
        switch (a.N) {                                              // instantiated agent counts (n^k for n = 2 .. 8)
            case 3: case 4: case 5: case 6: case 7: case 8: case 9: case 16: case 25: case 27: case 32: break;
            default: return false;
        }
        if (b->landmarks) return false;                             // landmark tracking: tile kernel
    }
    return warp_common_ok<T>(p, b);
}

// formation_hd_partial_env / formation_hd_partial_range_env on the warp-autonomous kernel (fg_warp_lm.cuh)
template <typename T>
bool lm_warp_ok(const fg::KArgs<T>& a, int scenario, const fg_params* p, const fg_buffers* b) {
    if (scenario != FG_SCENARIO_HD_PARTIAL && scenario != FG_SCENARIO_HD_PARTIAL_RANGE &&
        scenario != FG_SCENARIO_HD_OBSTACLE) return false;
    if (a.N < 3 || a.N > 9 || !b->landmarks || !b->obs) return false;
    return warp_common_ok<T>(p, b);
}

// Per-scenario state: formation_hd_env reads ideal_shape / ideal_vel, every other scenario its landmarks
int check_state(const fg_buffers* b, int scenario, const char* who) {
    if (scenario == FG_SCENARIO_HD && (!b->ideal_shape || !b->ideal_vel))
        return fail(FG_ERR_ARG, "%s(hd): ideal_shape/ideal_vel must be non-null", who);
    if (scenario != FG_SCENARIO_HD && !b->landmarks)
        return fail(FG_ERR_ARG, "%s: landmarks must be non-null for this scenario", who);
    return FG_OK;
}

// The observation pass without physics (k_step / k_step_obst, PHYS off) of fg_obs_reward, fg_final_obs, fg_obs_gather
template <typename T>
int launch_obs(const fg::KArgs<T>& a, int scenario, const fg_params* p, void* stream) {
    if (scenario == FG_SCENARIO_HD_OBSTACLE) return launch_obstacle<T, false>(a, stream);
    return launch<T, false, true>(a, scenario, p, stream);
}

// The observation pass on the E records of a state block (fg_final layout) into obs, in the EXT instantiation:
// fg_final_obs passes done (the rows of ended envs only), fg_obs_gather rows / R (slot b reads record rows[b] of R).
// reward, step, done, nan_flag, lmv stay NULL.
template <typename T>
int state_obs(const fg_params* p, const fg_final* s, void* obs, int scenario, int E, int N, int L, const uint8_t* done,
              const int64_t* rows, long long R, void* stream) {
    fg_buffers b;
    memset(&b, 0, sizeof(b));
    b.pos = s->pos; b.vel = s->vel; b.obs = obs;
    if (p && !p->silent) b.comm = s->comm;
    if (scenario == FG_SCENARIO_HD) { b.ideal_shape = s->ideal_shape; b.ideal_vel = s->ideal_vel; }
    else b.landmarks = s->landmarks;                                // (hd: no landmark side effect)
    fg::KArgs<T> a;
    int rc = fill_args<T>(a, p, &b, scenario, E, N, L, 0, 0, 0);
    if (rc) return rc;
    set_final<T>(a, s, p, scenario);
    a.fin_done = done; a.gth_rows = rows; a.gth_count = R;
    return launch_obs<T>(a, scenario, p, stream);
}

template <typename T>
int world_step_impl(const fg_params* p, const fg_buffers* b, int E, int N, uint64_t seed, uint32_t tick,
                    uint32_t env_offset, void* stream) {
    NvtxRange nvtx_("fg_world_step");
    fg::KArgs<T> a;
    if (p && b && p->num_obstacles > 0 && b->contact_pos)
        return fail(FG_ERR_ARG, "fg_world_step: contact_pos (World.cache_dists) is not supported with movable obstacles%s");
    if (p && p->num_obstacles > 0) {
        // World.step on a world with movable colliding landmarks (formation_hd_obs_env's obstacles)
        int rc = fill_args<T>(a, p, b, FG_SCENARIO_HD_OBSTACLE, E, N, p->num_landmarks, seed, tick, env_offset);
        if (rc) return rc;
        if (!b->pos || !b->vel || !b->act || !b->landmarks)
            return fail(FG_ERR_ARG, "fg_world_step: pos/vel/act/landmarks must be non-null%s");
        return launch_obstacle<T, true, false>(a, stream);
    }
    // the physics does not depend on the scenario; hd's N>=3 rule must not apply here
    int rc = fill_args<T>(a, p, b, FG_SCENARIO_BASIC, E, N, 1, seed, tick, env_offset);
    if (rc) return rc;
    if (!b->pos || !b->vel || !b->act) return fail(FG_ERR_ARG, "fg_world_step: pos/vel/act must be non-null%s");
    return launch<T, true, false>(a, FG_SCENARIO_BASIC, p, stream);
}

template <typename T>
int obs_reward_impl(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L, void* stream) {
    NvtxRange nvtx_("fg_obs_reward");
    fg::KArgs<T> a;
    int rc = fill_args<T>(a, p, b, scenario, E, N, L, 0, 0, 0);
    if (rc) return rc;
    if (!b->pos || !b->vel || !b->reward) return fail(FG_ERR_ARG, "fg_obs_reward: pos/vel/reward must be non-null%s");
    rc = check_state(b, scenario, "fg_obs_reward");
    if (rc) return rc;
    a.step = nullptr; a.done = nullptr; a.ep_return = nullptr; a.ep_coll = nullptr; a.stats = nullptr;
    return launch_obs<T>(a, scenario, p, stream);
}

// Terminal observations (fg_final_obs): the observation pass of fg_obs_reward (k_step / k_step_obst without PHYS) on the
// terminal block, in the EXT instantiation that skips CTAs without an ended env and writes no reward.
template <typename T>
int final_obs_impl(const fg_params* p, const fg_final* f, const uint8_t* done, void* obs, int scenario, int E, int N,
                   int L, void* stream) {
    NvtxRange nvtx_("fg_final_obs");
    if (!f) return fail(FG_ERR_ARG, "fg_final_obs: the terminal block must be non-null%s");
    int rc = check_final<T>(f, p, scenario, 1, 1, false, "fg_final_obs");
    if (rc) return rc;
    if (!done || !obs) return fail(FG_ERR_ARG, "fg_final_obs: done / obs must be non-null%s");
    return state_obs<T>(p, f, obs, scenario, E, N, L, done, nullptr, 0, stream);
}

// Observations of sampled state records (fg_obs_gather): the same pass on a block of R records, in gather mode -- output
// slot b of the tile kernel reads record rows[b] (fg_kernels.cuh KArgs::gth_rows).
template <typename T>
int obs_gather_impl(const fg_params* p, const fg_final* s, long long R, const int64_t* rows, int B, void* obs,
                    int scenario, int N, int L, void* stream) {
    NvtxRange nvtx_("fg_obs_gather");
    if (!s) return fail(FG_ERR_ARG, "fg_obs_gather: the state block must be non-null%s");
    if (!rows || !obs) return fail(FG_ERR_ARG, "fg_obs_gather: rows / obs must be non-null%s");
    if (R < 1 || B < 1) return fail(FG_ERR_ARG, "fg_obs_gather: R and B must be >= 1%s");
    int rc = check_final<T>(s, p, scenario, 1, 1, false, "fg_obs_gather");
    if (rc) return rc;
    if (((uintptr_t)rows % sizeof(int64_t)) != 0) return fail(FG_ERR_ARG, "fg_obs_gather: rows must be 8-byte aligned%s");
    return state_obs<T>(p, s, obs, scenario, B, N, L, nullptr, rows, R, stream);   // E = B output slots
}

template <typename T>
int step_fused_impl(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L, int n_steps,
                    int random_actions, int auto_reset, uint64_t seed, uint32_t tick, uint32_t env_offset,
                    void* stream, const fg_targets* tg, const fg_final* fin) {
    NvtxRange nvtx_("fg_step_fused");
    int rc = check_targets<T>(tg, scenario, "fg_step_fused_targets");
    if (rc) return rc;
    rc = check_final<T>(fin, p, scenario, auto_reset, n_steps, true, "fg_step_fused_final");
    if (rc) return rc;
    fg::KArgs<T> a;
    rc = fill_args<T>(a, p, b, scenario, E, N, L, seed, tick, env_offset);
    if (rc) return rc;
    set_targets<T>(a, tg);
    set_final<T>(a, fin, p, scenario);
    if (!b->pos || !b->vel || !b->reward || !b->done || !b->step)
        return fail(FG_ERR_ARG, "fg_step_fused: pos/vel/reward/done/step must be non-null%s");
    if (!random_actions && !b->act) return fail(FG_ERR_ARG, "fg_step_fused: act is null and random_actions == 0%s");
    if (n_steps < 1) return fail(FG_ERR_ARG, "fg_step_fused: n_steps must be >= 1%s");
    if (n_steps > 1 && !random_actions)
        return fail(FG_ERR_ARG, "fg_step_fused: n_steps > 1 needs random_actions (one action set per call)%s");
    if (random_actions < 0 || random_actions > 2) return fail(FG_ERR_ARG, "fg_step_fused: random_actions must be 0, 1 or 2%s");
    if (random_actions && !p->silent)
        return fail(FG_ERR_ARG, "fg_step_fused: random_actions supports silent agents only%s");
    if (random_actions == 2 && !b->act)
        return fail(FG_ERR_ARG, "fg_step_fused: random_actions == 2 records the drawn actions in b->act (non-null)%s");
    rc = check_state(b, scenario, "fg_step_fused");
    if (rc) return rc;
    a.n_steps = n_steps; a.random_actions = random_actions; a.auto_reset = auto_reset;
    if (warp_path_ok<T>(a, scenario, p, b)) {
        cudaStream_t st = (cudaStream_t)stream;
        if (scenario == FG_SCENARIO_BASIC) return launch_warp<T, 3, fg::kScnBasic>(a, st);
        switch (N) {
            case 3: return launch_warp<T, 3>(a, st);
            case 4: return launch_warp<T, 4>(a, st);
            case 5: return launch_warp<T, 5>(a, st);
            case 6: return launch_warp<T, 6>(a, st);
            case 7: return launch_warp<T, 7>(a, st);
            case 8: return launch_warp<T, 8>(a, st);
            case 9: return launch_warp<T, 9>(a, st);
            case 16: return launch_warp<T, 16>(a, st);
            case 25: return launch_warp<T, 25>(a, st);
            case 32: return launch_warp<T, 32>(a, st);
            default: return launch_warp<T, 27>(a, st);
        }
    }
    if (lm_warp_ok<T>(a, scenario, p, b)) {
        rc = fgabi::launch_lm_warp(a, scenario, (cudaStream_t)stream);
        if (rc <= 0) return rc;                                     // (1: no instantiation -> tile kernel)
    }
    if (scenario == FG_SCENARIO_HD_OBSTACLE) return launch_obstacle<T, true>(a, stream);
    return launch<T, true, true>(a, scenario, p, stream);
}

template <typename T>
int reset_impl(const fg_params* p, const fg_buffers* b, int scenario, int E, int N, int L, const uint8_t* mask,
               uint64_t seed, uint32_t tick, uint32_t env_offset, void* stream, const fg_targets* tg) {
    NvtxRange nvtx_("fg_reset");
    int rc = check_targets<T>(tg, scenario, "fg_reset_targets");
    if (rc) return rc;
    fg::KArgs<T> a;
    rc = fill_args<T>(a, p, b, scenario, E, N, L, seed, tick, env_offset);
    if (rc) return rc;
    set_targets<T>(a, tg);
    if (!b->pos || !b->vel) return fail(FG_ERR_ARG, "fg_reset: pos/vel must be non-null%s");
    rc = check_state(b, scenario, "fg_reset");
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = (E + 127) / 128;
    if (scenario == FG_SCENARIO_HD) fg::k_reset<T, fg::kScnHD><<<grid, 128, 0, st>>>(a, mask);
    else if (scenario == FG_SCENARIO_HD_OBSTACLE) fg::k_reset_obst<T><<<grid, 128, 0, st>>>(a, mask);
    else                            fg::k_reset<T, fg::kScnBasic><<<grid, 128, 0, st>>>(a, mask);
    return launch_status();
}

template <typename T>
int random_actions_impl(void* act, int E, int N, uint64_t seed, uint32_t tick, uint32_t env_offset,
                        const uint32_t* tick_dev, void* stream) {
    NvtxRange nvtx_("fg_random_actions");
    if (!act || E < 1 || N < 1) return fail(FG_ERR_ARG, "fg_random_actions: bad argument%s");
    if ((uint64_t)E * (uint64_t)N >= (1ull << 31)) return fail(FG_ERR_ARG, "E*N must be < 2^31%s");
    const uint32_t n = (uint32_t)E * (uint32_t)N;
    int grid = (int)((n + 255u) / 256u);
    if (grid > 148 * 32) grid = 148 * 32;                           // grid-stride beyond 32 CTAs per SM
    fg::k_random_actions<T><<<grid, 256, 0, (cudaStream_t)stream>>>((typename fg::Ops<T>::R2*)act, n, (uint32_t)N,
                                                                   seed, tick, env_offset, tick_dev);
    return launch_status();
}

template <typename T>
int pair_distances_impl(const void* ent, const void* size, int E, int M, void* vect, void* mag, uint8_t* coll, void* mind,
                        void* stream) {
    NvtxRange nvtx_("fg_pair_distances");
    typedef typename fg::Ops<T>::R2 R2;
    if (!ent || !size || !vect || !mag || !coll || !mind) return fail(FG_ERR_ARG, "fg_pair_distances: null pointer%s");
    if (E < 1 || M < 1 || M > FG_MAX_AGENTS + FG_MAX_LANDMARKS) return fail(FG_ERR_ARG, "fg_pair_distances: bad E or M%s");
    const size_t total = (size_t)E * M * M;
    int grid = (int)std::min<size_t>((total + 255) / 256, (size_t)148 * 16);
    fg::k_pair_distances<T><<<grid, 256, 0, (cudaStream_t)stream>>>((const R2*)ent, (const T*)size, E, M, (R2*)vect, (T*)mag,
                                                                    coll, (T*)mind);
    return launch_status();
}

// The reference's controller tree over N agents, n per layer: N = n^levels (the reference asserts log(len(obs))/log(n)
// is an integer, formation_gym/__init__.py:55-56; levels = 0 when it is not) and the multiplier log(M)/log(n) of each
// layer of M agents, top first (:78).
struct PolicyTree { int levels; double mult[fg::kPolicyMaxLevels]; };

PolicyTree policy_tree(int N, int n) {
    PolicyTree t{};
    int M = N;
    while (M > 1 && M % n == 0) { M /= n; ++t.levels; }
    if (M != 1 || t.levels < 1 || t.levels > fg::kPolicyMaxLevels) return PolicyTree{};
    M = N;
    for (int l = 0; l < t.levels; ++l) { t.mult[l] = std::log((double)M) / std::log((double)n); M /= n; }
    return t;
}

template <typename T>
int policy_bfs_impl(const void* pos, const void* shape, const void* ivel, void* act, int E, int N, int n,
                    void* stream) {
    NvtxRange nvtx_("fg_policy_bfs");
    typedef typename fg::Ops<T>::R2 R2;
    if (!pos || !shape || !ivel || !act) return fail(FG_ERR_ARG, "fg_policy_bfs: null pointer%s");
    if (E < 1 || N < 1 || N > FG_MAX_AGENTS) return fail(FG_ERR_ARG, "fg_policy_bfs: bad E or N%s");
    if (n < 2 || n > fg::kPolicyMaxFan) return fail(FG_ERR_ARG, "fg_policy_bfs: num_agents_per_layer must be in [2, 8]%s");
    const PolicyTree tree = policy_tree(N, n);
    const int levels = tree.levels;
    if (!levels)
        return fail(FG_ERR_ARG, "fg_policy_bfs: N must be a power of num_agents_per_layer ('Observation shape error!')%s");
    fg::PArgs<T> a;
    memset(&a, 0, sizeof(a));
    a.pos = (const R2*)pos; a.shape = (const R2*)shape; a.ivel = (const R2*)ivel; a.act = (R2*)act;
    a.E = E; a.N = N; a.n = n; a.levels = levels; a.EPC = fg::kBlock / N; a.magic_n = magic_for(N);
    int M = N;
    for (int l = 0; l < levels; ++l) {
        a.mult[l] = (T)tree.mult[l];
        a.lev_M[l] = M; a.lev_nxt[l] = M / n; a.lev_nlead[l] = N / (M / n);
        a.mg_M[l] = magic_for(M); a.mg_nxt[l] = magic_for(M / n); a.mg_nlead[l] = magic_for(N / (M / n));
        M /= n;
    }
    const size_t smem = (size_t)4 * a.EPC * N * sizeof(R2);
    const int grid = (E + a.EPC - 1) / a.EPC;
    cudaStream_t st = (cudaStream_t)stream;
    // compile-time tree shapes for the reference's own sizes (README.md:31-51: groups of 3, up to 3^5 agents; test.py
    // --num-layer) and the binary / quaternary trees up to 32 / 16 agents; run-time shape otherwise
    const int key = n * 16 + levels;
    switch (key) {
#define FG_POLICY_CASE(NF_, LV_) case NF_ * 16 + LV_: fg::k_policy_bfs<T, NF_, LV_><<<grid, fg::kBlock, smem, st>>>(a); break;
        FG_POLICY_CASE(3, 1) FG_POLICY_CASE(3, 2) FG_POLICY_CASE(3, 3) FG_POLICY_CASE(3, 4) FG_POLICY_CASE(3, 5)
        FG_POLICY_CASE(2, 2) FG_POLICY_CASE(2, 3) FG_POLICY_CASE(2, 4) FG_POLICY_CASE(2, 5)
        FG_POLICY_CASE(4, 1) FG_POLICY_CASE(4, 2) FG_POLICY_CASE(5, 1) FG_POLICY_CASE(5, 2)
#undef FG_POLICY_CASE
        default:
            switch (n) {                                            // compile-time fan-out for the usual group sizes
                case 2: fg::k_policy_bfs<T, 2><<<grid, fg::kBlock, smem, st>>>(a); break;
                case 3: fg::k_policy_bfs<T, 3><<<grid, fg::kBlock, smem, st>>>(a); break;
                case 4: fg::k_policy_bfs<T, 4><<<grid, fg::kBlock, smem, st>>>(a); break;
                case 5: fg::k_policy_bfs<T, 5><<<grid, fg::kBlock, smem, st>>>(a); break;
                default: fg::k_policy_bfs<T, 0><<<grid, fg::kBlock, smem, st>>>(a); break;
            }
    }
    return launch_status();
}

}  // namespace

