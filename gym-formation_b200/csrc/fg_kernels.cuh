// fg_kernels.cuh -- the fused MPE step kernel (sm_100a) and its small companions.
//
// One CTA owns a TILE of EPC = floor(256 / N) consecutive envs; thread t <-> (local env t / N,
// agent t % N), so N = 3, 9, 27, 81, 243 fill 255, 252, 243, 243, 243 of the 256 lanes.  A tile's
// state (pos, vel, ideal shape / landmarks, comm) is staged in shared memory with coalesced
// 8-byte (fp32) / 16-byte (fp64) loads; the O(N^2) pair loops read the other agents of the same
// env from shared memory (same address across the lanes of an env -> broadcast, no conflicts).
// Phases of one env step (reference file:line for each in the code):
//   load -> [sync] -> action force + pairwise contact force (OLD positions) + integrate
//        -> [sync] -> centroid / collision count / Hausdorff partials (NEW positions)
//        -> [sync] -> rewards, done, episode statistics -> [auto-reset, sync]
//        -> observation rows emitted as ONE contiguous, fully coalesced span per tile.
// The observation tensor is 24 N^2 of the 24 N^2 + 53 N + 16 algorithmic bytes per env-step, so
// the kernel is an HBM-store-bound obs writer with the physics riding along (DESIGN.md).
#pragma once
#include "fg_math.cuh"
#include "fg_pairs.cuh"

namespace fg {

constexpr int kBlock = 256;
constexpr int kMaxWalls = 8;
constexpr int kScnHD = 0;
constexpr int kScnBasic = 1;
constexpr int kScnPartial = 2;      // formation_hd_partial_env: landmarks absolute, the next num_obs agents
constexpr int kScnRange = 3;        // formation_hd_partial_range_env: landmarks absolute, other_pos clipped to a range

template <typename T> struct WallT {
    int orient, hard;
    T axis_pos, end0, end1, width;
};

template <typename T> struct KArgs {
    typedef typename Ops<T>::R2 R2;
    // buffers (see include/formation_gym_b200.h fg_buffers)
    R2* pos; R2* vel; const R2* act; R2* comm;
    R2* shape; R2* ivel; R2* lm;
    int32_t* step;
    R2* obs; T* reward; T* indiv; uint8_t* done;
    T* ep_return; int32_t* ep_coll; double* stats;
    const T* a_mass; const T* a_size; const T* a_accel; const T* a_vmax;
    // sizes
    int E, N, L, EPC, IPR;           // IPR = R2 items per observation row (hd 3N; basic 2+L+2(N-1))
    uint32_t magic_n, magic_ipr;     // fastdiv magics for N and IPR
    uint32_t magic_l, magic_np;      // ... for L (landmark loops) and roundup(N, 32)
    int act_r2;                      // R2 elements per agent in act (1 silent, 2 with comm action)
    // params in T
    T dt, keep, cforce, margin, size, mass, vmax, u_noise, c_noise;
    T sens0;                         // environment.py:218 sensitivity (5.0)
    T accel;                         // scalar Entity.accel, used iff has_accel
    T sens, gain;                    // effective scalars: sens = has_accel ? accel : sens0; gain = has_accel ? mass*accel : mass
    T cut2;                          // (2*size + kcut*margin)^2 : contact early-out (uniform sizes)
    T kcut;
    T rthr, rthr2_hi;                // reward collision threshold and its guarded square
    int has_accel, has_vmax, collide, silent, world_length, n_walls, prescaled;
    int mass_one;                    // mass == 1: F / m is exact without the division
    int row_tma;                     // tile kernel: long hd rows leave through TMA bulk stores (see k_step)
    int row_nbuf;                    // OM == 2: staging buffers per warp (2; 1 when that lets one more CTA fit per SM)
    int row_chunk, row_chunk_log2;   // OM == 2, chunked writer: rows per shared-memory image (power of two; 0 = per-row pieces)
    int row_early;                   // OM == 2, fp32, odd N, 16-byte aligned obs: rows leave as aligned bulk pieces, the
                                     // static 2/3 before the physics and the dynamic 1/3 before the reward pass
    int fast_pairs;                  // tile kernel: packed pair loops of fg_pairs.cuh (N >= 32; fp32 hd uniform only)
    int cells;                       // fast pairs: near partners from hashed cell lists instead of the O(N^2) filters
    int cell_shift;                  // 32 - log2(buckets per env)
    unsigned cell_off;               // byte offset of the cell-list region in dynamic shared memory
    float cell_inv_old, cell_inv_new;   // 1 / cell edge: contact cut-off (old positions), reward collision (new)
    R2* lmv;                         // obstacle scenario: landmark velocities [E,L,2] (obstacle entries used)
    int n_obst;                      // obstacle scenario: the last n_obst landmarks are movable colliding obstacles
    T osize, omass, ofloor, ofall;   // obstacle size / mass, floor y and fall velocity of the reward hook's rule
    int num_obs;                     // partial: observed neighbours (formation_hd_partial_env.py:15,53)
    T obs_range;                     // range: clip bound of other_pos (formation_hd_partial_range_env.py:15,53)
    int n_steps, random_actions, auto_reset;
    int pf_dist;                     // warp kernel: > 0 = L2 prefetch of the state two spans ahead (see fg_warp.cuh)
    uint64_t seed; uint32_t tick; uint32_t env_offset;
    uint32_t* tick_dev;              // (opt) [2]: device tick added to `tick`, arrival counter (CUDA graphs)
    const R2* cpos;                  // (opt) [E,N,2] World.cache_dists: positions the contact forces are computed from
    uint8_t* nan_flag;               // (opt) [E]: set to 1 (never cleared) when the env holds a non-finite position (Q9)
    T pol_mult[8];                   // fused device controller (fg_warp.cuh, POL): log(M)/log(n) per BFS layer, top first
    WallT<T> walls[kMaxWalls];
    // formation_hd_env target bank (fg_targets; read only by the reset blocks): tgt_count = K tasks, 0 = no bank
    const R2* tgt_shape;             // [K,N] raw shapes, replacing the kResetLandmark draw
    const R2* tgt_vel;               // (opt) [K] ideal velocities, replacing the kResetIdealVel draw
    const int32_t* tgt_index;        // (opt) [E] task per env; out of [0, K) = draw
    int tgt_count;
    // terminal block (fg_final; written only by the reset blocks of the EXT instantiations): fin_pos == NULL = none.
    // fg_final_obs reads it back as the state (pos / vel / ...) and fin_done as the mask of ended envs.
    R2* fin_pos; R2* fin_vel; R2* fin_comm;
    R2* fin_shape; R2* fin_ivel; R2* fin_lm;
    const uint8_t* fin_done;         // fg_final_obs: done [E,N] of the step
    // gather mode of the observation pass (fg_obs_gather; read only by the EXT && !PHYS instantiations): the state is a
    // block of gth_count records (fin_* == pos / vel / ... shaped [R, ...]) and output slot b takes record gth_rows[b];
    // a slot whose index is outside [0, gth_count) reads nothing and gets NaN state.  gth_rows == NULL = off.
    const int64_t* gth_rows;
    long long gth_count;
};

// An instantiation with the reset extension (template flag EXT) runs when a target bank, a terminal block or a gather
// row list is set.
template <typename T>
__host__ __device__ __forceinline__ bool reset_ext(const KArgs<T>& a) {
    return a.tgt_count > 0 || a.fin_pos != nullptr || a.gth_rows != nullptr;
}

// Gather mode: record of output slot b, or -1 when its index names no record (then the slot reads nothing).
template <typename T>
__device__ __forceinline__ long long gather_record(const KArgs<T>& a, int b) {
    const long long r = a.gth_rows[b];
    return (r >= 0 && r < a.gth_count) ? r : -1;
}

// Task of env e (global id ge) at a reset with tick tk: tgt_index[e] when it names an entry of the bank, else
// drawn uniformly from Philox.  Only called when tgt_count > 0.
template <typename T>
__device__ __forceinline__ uint32_t target_task(const KArgs<T>& a, int e, uint32_t ge, uint32_t tk) {
    const uint32_t K = (uint32_t)a.tgt_count;
    if (a.tgt_index) {
        const int32_t k = a.tgt_index[e];
        if (k >= 0 && (uint32_t)k < K) return (uint32_t)k;
    }
    return __umulhi(philox(a.seed, ge, 0u, tk, kResetTarget).x, K);
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}

// One contiguous piece of an observation row, smem image -> HBM: the 16-byte-aligned middle as a TMA
// bulk store (cp.async.bulk, L2 evict_first; the caller commits the group), an odd 8-byte head / tail
// item as plain stores.  `img` holds the piece at the same offset modulo 16 as `dst`.
// Called by a whole warp: lane 0 issues the bulk copy, lanes 1 and 2 the head / tail items.
template <typename R2>
__device__ __forceinline__ void row_piece_store(R2* dst, const R2* img, uint32_t bytes, int lane) {
    const uint32_t head = min((uint32_t)((16u - ((uint32_t)(uintptr_t)dst & 15u)) & 15u), bytes);
    const uint32_t mid = (bytes - head) & ~15u;
    const uint32_t tail = bytes - head - mid;
    if (lane == 0) {
        if (mid) {
            uint64_t pol;
            asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;"
                         :: "l"(reinterpret_cast<unsigned char*>(dst) + head),
                            "r"(smem_u32(reinterpret_cast<const unsigned char*>(img) + head)), "r"(mid), "l"(pol)
                         : "memory");
        }
    } else if (lane == 1) {
        if (head) dst[0] = img[0];
    } else if (lane == 2) {
        if (tail) { const uint32_t it = (head + mid) / (uint32_t)sizeof(R2); dst[it] = img[it]; }
    }
}

// Device-side tick for CUDA-graph replays: every launch reads tick_dev[0] at its start; the LAST
// arriving participant (CTA or warp) of a stepping kernel advances it by the number of env steps
// the launch performed and re-arms the arrival counter tick_dev[1].
__device__ __forceinline__ void tick_arrive(uint32_t* tick_dev, unsigned participants, int n_steps, bool leader) {
    if (tick_dev && leader) {
        __threadfence();
        if (atomicAdd(&tick_dev[1], 1u) == participants - 1u) {
            tick_dev[1] = 0u;
            tick_dev[0] += (uint32_t)n_steps;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Contact cut-off of an env (DESIGN.md "contact cut-off").  Every pair loop skips a pair when its squared distance
// passes !(d2 >= cut2) -- NaN distances stay, but d2 = +inf would be dropped, where the reference (no cut-off,
// core.py:304-312) turns it into dist = inf, pen = 0 and force = 0 * inf / inf = NaN.  So an env with a non-finite
// old position of a colliding entity sends every pair to contact_force: through a NaN cut-off (env_cut2: k_lm_warp,
// k_step_obst) or, off the hot pair loops, through its near mask (k_hd_warp) or an all-pairs loop (k_step).  Finite
// envs keep the plain cut-off and their exact results.
template <typename T>
__device__ __forceinline__ bool nonfinite2(T x, T y) { return !(fabs(x) < (T)INFINITY) || !(fabs(y) < (T)INFINITY); }

template <typename R2>
__device__ __forceinline__ bool any_nonfinite(const R2* p, int n) {
    bool bad = false;
    for (int j = 0; j < n; ++j) bad |= nonfinite2(p[j].x, p[j].y);
    return bad;
}

template <typename T>
__device__ __forceinline__ T env_cut2(T cut2, bool env_nonfinite) {
    return env_nonfinite ? Ops<T>::from_bits(~(typename Ops<T>::Bits)0 >> 1) : cut2;
}

// ------------------------------------------------------------------------------------------------
// get_entity_collision_force (core.py:289-322), both entities movable colliders (agents).
// (dx,dy) = p_a - p_b with a < b in entity order.  Returns `force` (core.py:312).
template <typename T>
__device__ __forceinline__ void contact_force(T dx, T dy, T dmin, T k, T cf, T* fx, T* fy, bool cached = false) {
    typedef Ops<T> O;
    // core.py:305 np.linalg.norm(delta_pos); with World.cache_dists the distance comes from
    // np.linalg.norm(cached_dist_vect, axis=2) (core.py:178,299-300): a plain sqrt(x*x + y*y), no dot-product FMA
    T dist = cached ? O::sqrt_(O::sq2(dx, dy)) : O::norm2(dx, dy);
    T tt = O::div(-O::sub(dist, dmin), k);                       // -(dist - dist_min)/k
    // np.logaddexp(0, tt): stable softplus (core.py:310): tt > 0 ? tt + log1p(exp(-tt)) : log1p(exp(tt)).
    // Both branches share log1p(exp(-|tt|)), evaluated once (bit-identical to either branch).
    const T lg = O::log1p_(O::exp_(-fabs(tt)));
    T sp = (tt > (T)0) ? O::add(tt, lg) : lg;
    T pen = O::mul(sp, k);
    *fx = O::mul(O::div(O::mul(cf, dx), dist), pen);             // contact_force*delta/dist*pen
    *fy = O::mul(O::div(O::mul(cf, dy), dist), pen);             // dist == 0 -> NaN, as reference
}

// get_wall_collision_force (core.py:325-362) on one entity
template <typename T>
__device__ __forceinline__ void wall_force(const WallT<T>& w, T px, T py, T size, T k, T cf, T* fx, T* fy) {
    typedef Ops<T> O;
    T prll = w.orient == 0 ? px : py;
    T perp = w.orient == 0 ? py : px;
    *fx = (T)0; *fy = (T)0;
    if (prll < O::sub(w.end0, size) || prll > O::add(w.end1, size)) return;    // :335-337
    T theta = (T)0, dmin;
    if (prll < w.end0 || prll > w.end1) {                                       // :338-346
        T past = prll < w.end0 ? O::sub(prll, w.end0) : O::sub(prll, w.end1);
        theta = O::asin_(O::div(past, size));
        T s, c; O::sincos_(theta, &s, &c);
        dmin = O::add(O::mul(c, size), O::mul((T)0.5, w.width));
    } else {
        dmin = O::add(size, O::mul((T)0.5, w.width));                           // :350
    }
    T delta = O::sub(perp, w.axis_pos);                                         // :353
    T dist = fabs(delta);
    T tt = O::div(-O::sub(dist, dmin), k);
    T sp = (tt > (T)0) ? O::add(tt, O::log1p_(O::exp_(-tt))) : O::log1p_(O::exp_(tt));
    T pen = O::mul(sp, k);                                                      // :357
    T fmag = O::mul(O::div(O::mul(cf, delta), dist), pen);                      // :358
    T s, c; O::sincos_(theta, &s, &c);
    T fperp = O::mul(c, fmag), fprll = O::mul(s, fabs(fmag));                   // :360-361
    if (w.orient == 0) { *fx = fprll; *fy = fperp; } else { *fx = fperp; *fy = fprll; }
}

// ------------------------------------------------------------------------------------------------
// The fused kernel.  PHYS: run World.step.  OBSREW: run observation/reward/done.  HET: per-agent
// mass/size/accel/max_speed arrays (otherwise the scalar fast path).
// OM selects the observation writer (one per instantiation keeps registers low): 0 = flat item loop
// (fallback), 1 = one warp per row with plain streaming stores, 2 = one warp per row, static row part
// bulk-stored from a shared image (hd, silent agents, long rows), 3 = short rows: own row per thread staged in
// shared memory, the whole tile leaves as one bulk store.
// FP: fast pair loops of fg_pairs.cuh (fp32, hd, uniform agents, N >= 32): structure-of-arrays partner
// data, packed FFMA2/FADD2/FMUL2 arithmetic, group filters, warp-shuffle centroid and reductions.
// EXT: the reset extension -- a target bank (KArgs::tgt_*, formation_hd_env) and / or a terminal block (KArgs::fin_*),
// both run-time tests inside.  Its own instantiation, so that the reset block of the product kernels -- and with it
// their register allocation -- is the same as without the features.  Without PHYS, EXT is fg_final_obs: the state is
// the terminal block, a CTA without an ended env (fin_done) exits at once, and no reward is written.
template <typename T, int SCN, bool PHYS, bool OBSREW, bool HET, int OM, bool FP, bool EXT = false>
__global__ void __launch_bounds__(kBlock, (OM == 3 && SCN == kScnBasic) ? 5 : (OM == 2 || OM == 3 || FP) ? 4 : 3) k_step(const __grid_constant__ KArgs<T> a) {
    typedef Ops<T> O;
    typedef typename O::R2 R2;
    typedef typename O::Bits Bits;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr bool FINOBS = EXT && !PHYS;

    const int N = a.N, EPC = a.EPC, L = a.L;
    const int nA = EPC * N;
    const int nS = (SCN == kScnHD) ? nA : EPC * L;
    // row-TMA region (OM == 2): per local env two images of the row's static part
    // [comm zeros (N-1) | ideal_shape (N) | ideal_vel], one per 16-byte phase, then one staging
    // buffer per warp for a row's dynamic part [p_vel | other_pos (N-1)].
    const int rt_img = 2 * N + 1;                     // items per static image incl. one pad item
    const int rt_dyn = (N + 3) & ~1;                  // items per staging buffer (16-byte multiple)
    R2* s_rt_img = reinterpret_cast<R2*>(smem_raw);
    R2* s_rt_dyn = s_rt_img + (OM == 2 ? 2 * rt_img * EPC : 0);
    // OM == 3: image of the whole tile's observation rows (own row per thread), + 2 items for the 16-byte phase
    const int img3_items = (OM == 3) ? ((EPC * N * a.IPR + 3) & ~1) : 0;
    if (OM == 3) s_rt_dyn = s_rt_img + img3_items;
    // FP: per local env, arrays of NP = roundup(N, 32) floats (16-byte aligned): old positions and
    // their squared norms, centred new positions and norms, centred ideal shape.
    const int NP = (N + 31) & ~31;
    const int NB = a.row_nbuf;
    float* f_base = (OM == 2 && a.row_chunk)
        ? reinterpret_cast<float*>(s_rt_img + ((a.row_chunk * a.IPR + 3) & ~1))
        : reinterpret_cast<float*>(s_rt_dyn + (OM == 2 ? NB * rt_dyn * (kBlock / 32) : 0));
    // Partner data as RECORDS of four partners (one address register + immediate offsets in the pair loops):
    // f_ro [EPC][NP/4] x {x[4], y[4], |p|^2[4]} of the old positions (contact filter),
    // f_rn [EPC][NP/4] x {cx[4], cy[4], |c|^2[4], sx[4], sy[4]} centred new positions and centred ideal shape.
    float* f_ro = f_base;
    float* f_rn = f_ro + 3 * EPC * NP;
    float* f_part = f_rn + 5 * EPC * NP;              // [EPC][8 warps][4]: partial sums of pos.xy, vel.xy
    const int NG = NP >> 2;                           // records per env
    auto RO = [&](int e_, int i_, int c_) -> float& { return f_ro[((e_ * NG + (i_ >> 2)) * 3 + c_) * 4 + (i_ & 3)]; };
    auto RN = [&](int e_, int i_, int c_) -> float& { return f_rn[((e_ * NG + (i_ >> 2)) * 5 + c_) * 4 + (i_ & 3)]; };
    R2* s_old = reinterpret_cast<R2*>(f_base + (FP ? 8 * EPC * NP + EPC * 32 : 0));   // positions the contact force reads
    R2* s_new = s_old + nA;                           // positions after integration
    R2* s_v = s_new + nA;                             // velocities after integration
    R2* s_s = s_v + nA;                               // hd: centred ideal shape; basic: landmarks
    R2* s_c = s_s + nS;                               // comm state
    R2* s_iv = s_c + nA;                              // hd: ideal velocity per env
    R2* s_mean = s_iv + EPC;                          // hd: [EPC][2] centroid, mean velocity
    R2* s_cen = s_mean + 2 * EPC;                     // hd: centred new positions [nA]
    Bits* s_rowmax = reinterpret_cast<Bits*>(s_cen + ((SCN != kScnBasic) ? nA : 0));   // max of the Hausdorff minima
    T* s_lmin = reinterpret_cast<T*>(s_rowmax + EPC);         // basic: min_a |p_a - l_k| [EPC*L]
    T* s_het = s_lmin + ((SCN == kScnBasic) ? EPC * L : 0);   // HET: mass,size,sens,gain,vmax [5N]
    int* s_col = reinterpret_cast<int*>(s_het + (HET ? 5 * N : 0));
    int* s_dn = s_col + EPC;                                  // episode-end flag per local env
    int* s_bad = s_dn + EPC;                                  // env has a non-finite position (NaN quirk, Q9)
    unsigned* s_nmax = reinterpret_cast<unsigned*>(s_bad + EPC);   // FP: [2][EPC] max |p|^2 bits (old, centred new)
    // FP + cells: two hashed cell lists per env (old positions: contact cut-off; new positions: reward collision):
    // bucket heads [2][EPC][CB], chain links [2][EPC][NP], "env has a far / non-finite agent" flags [2][EPC]
    const int CB = 1 << (32 - a.cell_shift);
    float4* c_node = reinterpret_cast<float4*>(smem_raw + a.cell_off);       // [2][EPC][NP] chain nodes {x, y, next}
    int* c_head = reinterpret_cast<int*>(c_node + 2 * EPC * NP);             // [2][EPC][CB] bucket heads
    int* c_far = c_head + 2 * EPC * CB;                                      // [2][EPC]
    __shared__ double s_stat[4];                              // episode statistics of this CTA's envs
    if (threadIdx.x < 4) s_stat[threadIdx.x] = 0.0;

    const int t = threadIdx.x;
    const uint32_t tick0 = a.tick + (a.tick_dev ? a.tick_dev[0] : 0u);   // read before the first barrier
    const int tile0 = blockIdx.x * EPC;                       // first env of this tile
    const int le = (int)fastdiv((uint32_t)t, a.magic_n);
    const int i = t - le * N;
    const int e = tile0 + le;
    const bool active = (t < nA) && (e < a.E);
    const int nvalid = min(EPC, a.E - tile0);                 // envs of this tile that exist
    const size_t g = (size_t)e * N + i;                       // global agent index
    const uint32_t ge = a.env_offset + (uint32_t)e;           // global env id (RNG counter)

    // Gather mode (FINOBS with gth_rows): this thread reads agent i of record rec = gth_rows[e] (64-bit addressing: a
    // block of T x E records passes 2^32 bytes quickly); rec < 0 names no record: NaN state, nothing is read.  The rows
    // still leave at the tile position e, so the observation writers below are those of fg_final_obs.
    long long rec = e;
    if constexpr (FINOBS) {
        if (a.gth_rows) {
            if (active) rec = gather_record(a, e);
        } else if (!__syncthreads_or(t < nvalid && a.fin_done[(size_t)(tile0 + t) * N] != 0)) {
            return;                                           // rows only where an episode ended (EPC <= kBlock)
        }
    }
    const size_t gs = FINOBS ? (size_t)rec * N + i : g;       // agent index of the state read
    const bool miss = FINOBS && rec < 0;
    const R2 nan2 = O::make((T)NAN, (T)NAN);

    if (HET) {
        for (int q = t; q < N; q += kBlock) {
            T m = a.a_mass ? a.a_mass[q] : a.mass;
            T acc = a.a_accel ? a.a_accel[q] : (T)-1;
            s_het[q] = m;
            s_het[N + q] = a.a_size ? a.a_size[q] : a.size;
            // environment.py:218-221 (sensitivity := accel) and core.py:235-236 (gain mass*accel)
            if (!a.a_accel && a.has_accel) acc = a.accel;
            s_het[2 * N + q] = a.prescaled ? (T)1 : (acc >= (T)0 ? acc : a.sens0);
            s_het[3 * N + q] = acc >= (T)0 ? O::mul(m, acc) : m;
            s_het[4 * N + q] = a.a_vmax ? a.a_vmax[q] : (a.has_vmax ? a.vmax : (T)-1);
        }
    }

    if (FP) {
        // neutral pad entries (never a candidate, never a minimum); the live entries are written below
        for (int q = t; q < EPC * NP; q += kBlock) {
            const int qe = (int)fastdiv((uint32_t)q, a.magic_np), qi = q - qe * NP;
            if (qi >= N) {
                RO(qe, qi, 0) = 0.f; RO(qe, qi, 1) = 0.f; RO(qe, qi, 2) = INFINITY;
                RN(qe, qi, 0) = 1e18f; RN(qe, qi, 1) = 1e18f; RN(qe, qi, 2) = INFINITY;
                RN(qe, qi, 3) = 1e18f; RN(qe, qi, 4) = 1e18f;
            }
        }
        if (t < 2 * EPC) s_nmax[t] = 0u;
        __syncthreads();
    }

    // ---- load the tile (coalesced: consecutive threads <-> consecutive agents of consecutive envs)
    R2 p = O::make((T)0, (T)0), v = p, u = p, uc = p;
    int stp = 0;
    if (active) {
        p = miss ? nan2 : a.pos[gs];
        v = miss ? nan2 : a.vel[gs];
        if (PHYS && !a.random_actions) {
            u = a.act[g * a.act_r2];
            if (a.act_r2 > 1) uc = a.act[g * a.act_r2 + 1];
        }
        if (PHYS) s_old[t] = a.cpos ? a.cpos[g] : p; else { s_new[t] = p; s_v[t] = v; }
        if (OBSREW) {
            if (SCN == kScnHD) {
                const R2 S0 = miss ? nan2 : a.shape[gs];
                s_s[t] = S0;
                if constexpr (FP) { RN(le, i, 3) = (float)S0.x; RN(le, i, 4) = (float)S0.y; }
                if constexpr (OM == 2) {
                    if (a.row_early && !a.row_chunk) {   // static row images [comm zeros (N-1) | ideal_shape (N) | ideal_vel], both phases
                        R2* im0 = s_rt_img + (size_t)le * 2 * rt_img;
                        R2* im1 = im0 + rt_img;
                        // (fg_obs_gather: a slot without a record gets NaN in place of the comm zeros too)
                        const R2 cz = miss ? nan2 : O::make((T)0, (T)0);
                        im0[N - 1 + i] = S0; im1[N - 1 + i] = S0;
                        if (i < N - 1) { im0[i] = cz; im1[i] = cz; }
                    }
                }
            }
            if (a.step) stp = a.step[e];
            if (!PHYS) s_c[t] = miss ? nan2 : (a.comm ? a.comm[gs] : O::make((T)0, (T)0));
        }
    }
    if (OBSREW) {
        if (SCN == kScnHD) {
            if (active && i == 0) {
                const R2 iv0 = miss ? nan2 : a.ivel[FINOBS ? (size_t)rec : (size_t)e];
                s_iv[le] = iv0;
                if constexpr (OM == 2) {
                    if (a.row_early && !a.row_chunk) {
                        R2* im0 = s_rt_img + (size_t)le * 2 * rt_img;
                        im0[2 * N - 1] = iv0; im0[rt_img + 2 * N - 1] = iv0;
                    }
                }
            }
        } else if (FINOBS && a.gth_rows) {
            for (int q = t; q < nvalid * L; q += kBlock) {
                const int qe = (int)fastdiv((uint32_t)q, a.magic_l), k = q - qe * L;
                const long long r = gather_record(a, tile0 + qe);
                s_s[q] = r < 0 ? nan2 : a.lm[(size_t)r * L + k];
            }
        } else {
            for (int q = t; q < nvalid * L; q += kBlock) s_s[q] = a.lm[(size_t)tile0 * L + q];
        }
    }

    // FP: a warp spans at most two envs (N >= 32): A = the env of lane 0, B = the next one
    const int lane_ = t & 31, wp_ = t >> 5;
    const int leA = __shfl_sync(0xffffffffu, le, 0);
    const bool inA = active && le == leA, inB = active && le != leA;
    const unsigned maskA = __ballot_sync(0xffffffffu, inA), maskB = __ballot_sync(0xffffffffu, inB);
    // max / sum over the lanes of my env in this warp, then ONE shared-memory atomic per (warp, env)
    auto env_atomic_max = [&](unsigned* dst, unsigned val) {
        if (inA) { unsigned m = __reduce_max_sync(maskA, val); if (lane_ == __ffs(maskA) - 1) atomicMax(&dst[le], m); }
        if (inB) { unsigned m = __reduce_max_sync(maskB, val); if (lane_ == __ffs(maskB) - 1) atomicMax(&dst[le], m); }
    };
    auto env_atomic_add = [&](int* dst, int val) {
        if (inA) { int m = __reduce_add_sync(maskA, val); if (m && lane_ == __ffs(maskA) - 1) atomicAdd(&dst[le], m); }
        if (inB) { int m = __reduce_add_sync(maskB, val); if (m && lane_ == __ffs(maskB) - 1) atomicAdd(&dst[le], m); }
    };

    // Chunked row writer (OM == 2, a.row_chunk = RC rows per chunk, a power of two): the CTA stages RC whole rows
    // [p_vel | other_pos | comm zeros | ideal_shape | ideal_vel] (formation_hd_env.py:52-59) in ONE shared-memory image --
    // 256 / RC consecutive threads share a row and walk its segments with plain strided loops -- and the chunk, RC consecutive rows of the [E,N,6N] tensor, leaves as ONE TMA bulk store of
    // RC * 24N bytes (a lone 8-byte head / tail item by plain stores when the tile starts on an odd 8-byte slot).  The
    // per-row writer above it spends ~200 warp instructions per row on bookkeeping and two small bulk stores
    // (profiles/r02_hd_n81: 77 % issue-active, 656 B + 1296 B pieces); this one ~50 and 1 / RC of a 31 KB store.
    // (Two half-size images so that a chunk can be filled while the previous one is read were measured slower for every
    // N: 0.61 vs 0.70 of the HBM peak at N = 20, 0.73 vs 0.79 at N = 40, 0.61 vs 0.74 at N = 64 -- the chunk size matters more.)
    auto rows_chunked = [&]() {
        const int RC = a.row_chunk, NS = kBlock >> a.row_chunk_log2;
        // consecutive threads <-> consecutive items of one row (conflict-free for every N; rows along the lanes instead
        // put rows 3N items apart into the same banks for even N: 0.27 of the HBM peak at N = 64)
        const int sl = t & (NS - 1), r = t / NS;
        const int nrows = nvalid * N, IPR = a.IPR;
        R2* out0 = a.obs + (size_t)tile0 * N * IPR;
        R2* img = s_rt_img + (((uint32_t)(uintptr_t)out0 & 15u) ? 1 : 0);           // same 16-byte phase as the tile
        const R2 zero2 = O::make((T)0, (T)0);
        for (int c0 = 0; c0 < nrows; c0 += RC) {
            const int nr = min(RC, nrows - c0);
            if (c0 > 0) {                                   // the image is still being read by the previous chunk's copy
                if (t == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                __syncthreads();
            }
            if (r < nr) {
                const int R = c0 + r;
                const int rle = (int)fastdiv((uint32_t)R, a.magic_n), ri = R - rle * N;
                const R2* P = s_new + rle * N;
                const R2* S = s_s + rle * N;
                const R2 pi = P[ri];
                R2* row = img + (size_t)r * IPR;
                for (int m = sl; m < N - 1; m += NS) {
                    const R2 pj = P[m + (m >= ri)];
                    row[1 + m] = O::make(O::sub(pj.x, pi.x), O::sub(pj.y, pi.y));   // other_pos (formation_hd_env.py:55)
                    // comm of the others (silent: zeros; fg_obs_gather reads s_c, NaN for a slot without a record).
                    // (if constexpr: the product instantiations' lambda must not capture s_c)
                    R2 cz = zero2;
                    if constexpr (FINOBS) cz = s_c[rle * N + m + (m >= ri)];
                    row[N + m] = cz;
                }
                for (int m = sl; m < N; m += NS) row[2 * N - 1 + m] = S[m];         // ideal_shape.flatten()
                if (sl == 0) { row[0] = s_v[R]; row[3 * N - 1] = s_iv[rle]; }       // p_vel, ideal_vel
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncthreads();
            if (t < 32) {
                row_piece_store<R2>(out0 + (size_t)c0 * IPR, img, (uint32_t)((size_t)nr * IPR * sizeof(R2)), t);
                if (t == 0) asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
        }
    };

    for (int ts = 0; ts < a.n_steps; ++ts) {
        if (OBSREW && t < EPC) { s_rowmax[t] = 0; s_col[t] = 0; s_bad[t] = 0; if (FP) s_nmax[EPC + t] = 0u; }
        float n_old = 0.f;
        if constexpr (FP) {
            if (a.cells) {
                for (int q = t; q < 2 * EPC * CB; q += kBlock) c_head[q] = -1;
                if (t < 2 * EPC) c_far[t] = 0;
            } else if (PHYS) {                                  // partner arrays of the contact filter
                n_old = (float)p.x * (float)p.x + (float)p.y * (float)p.y;
                if (active) { RO(le, i, 0) = (float)p.x; RO(le, i, 1) = (float)p.y; RO(le, i, 2) = n_old; }
                env_atomic_max(s_nmax, __float_as_uint(n_old));
            }
            if (t < EPC * 32) f_part[t] = 0.f;
        }
        // Early observation rows (OM == 2, a.row_early): unless an env of this tile ends its episode in this
        // step (then the rows must show the RESET state and everything is written after the reset, below),
        // the rows are sent right after the physics, BEFORE the reward pass, and drain under it.  (Sending the
        // static 2/3 even earlier, before the physics, was measured slower: 327 vs 260 us per 1024 envs of
        // 243 agents -- the burst fills the SM's TMA queue and the warps block on issuing; round 2 repeated it on
        // every second CTA only, so that the others compute meanwhile: 293 vs 244 us, still slower; delaying the
        // k-th resident CTA of an SM by k x 1.5 .. 8 us so that not all CTAs of the first wave are in their HBM-idle
        // load + physics phase together: 263 .. 285 vs 252 us, slower too.  The launch costs a fixed ~20-27 us on top of
        // 0.215 us per env (linear fit 592 .. 4096 envs): first-row latency plus the drain of the last CTAs.  Splitting
        // an env's rows over two CTAs that both run the physics would not shrink it: with every CTA writing only HALF
        // of its rows (timing experiment) the fit is 24.4 us + 0.111 us per CTA, so 1024 envs as 2048 half-CTAs cost
        // 245.6 us against 241.1 us now.)
        // The barrier also tells whether some env of the tile holds a non-finite old position (only then do the
        // threads scan their env for one, see env_cut2).  s_old[t] is this thread's own write.
        bool obad = false;
        if (PHYS && active && a.collide) { const R2 q = a.cpos ? s_old[t] : p; obad = nonfinite2(q.x, q.y); }
        bool early = false, tile_nf;
        if constexpr (OM == 2 && sizeof(R2) == 8) {
            if (a.obs && a.row_early) {
                const bool will_reset = active && a.auto_reset && a.step && (stp + 1 >= a.world_length);
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // images (generic proxy) -> async proxy
                tile_nf = __syncthreads_or((will_reset || obad) ? 1 : 0) != 0;   // rare: then ask both questions
                if (tile_nf) {
                    early = !__syncthreads_or(will_reset ? 1 : 0);
                    tile_nf = __syncthreads_or(obad ? 1 : 0) != 0;
                } else {
                    early = true;
                }
            } else {
                tile_nf = __syncthreads_or(obad ? 1 : 0) != 0;
            }
        } else {
            tile_nf = __syncthreads_or(obad ? 1 : 0) != 0;
        }
        // my env holds a non-finite old position: every pair goes to the contact force, in the loop below
        const bool env_nf = tile_nf && active && any_nonfinite(s_old + le * N, N);

        CellPos cpos = {0, 0, 1, 1};                                        // FP + cells: my cell (old positions)
        if constexpr (FP && PHYS) {
            if (a.cells && a.collide) {
                if (active) cpos = cell_insert((float)p.x, (float)p.y, a.cell_inv_old, a.cell_shift, c_head + le * CB,
                                               c_node + le * NP, i, &c_far[le]);
                __syncthreads();
            }
        }
        // =============================== World.step (core.py:206-225) ===========================
        if (PHYS) {
            if (active) {
                if (a.random_actions) {                                     // test.py:20
                    U4 r = philox(a.seed, ge, (uint32_t)i, tick0 + (uint32_t)ts, kAction);
                    u = O::make(uniform_pm1<T>(r.x), uniform_pm1<T>(r.y));
                    if (a.random_actions == 2) const_cast<R2*>(a.act)[g] = u;   // recorded for the caller (replay buffer)
                }
                T m_i = HET ? s_het[i] : a.mass;
                T size_i = HET ? s_het[N + i] : a.size;
                T sens = HET ? s_het[2 * N + i] : a.sens;
                T gain = HET ? s_het[3 * N + i] : a.gain;
                // _set_action: u *= sensitivity (environment.py:216-221);
                // apply_action_force: F = gain * u + noise (core.py:232-236)
                T Fx = O::mul(gain, O::mul(u.x, sens));
                T Fy = O::mul(gain, O::mul(u.y, sens));
                if (a.u_noise > (T)0) {
                    U4 r = philox(a.seed, ge, (uint32_t)i, tick0 + (uint32_t)ts, kUNoise);
                    T n0, n1; normal_pair<T>(r.x, r.y, &n0, &n1);
                    Fx = O::add(Fx, O::mul(n0, a.u_noise));
                    Fy = O::add(Fy, O::mul(n1, a.u_noise));
                }
                // apply_environment_force (core.py:240-254): pairs a<b; contributions reach agent
                // i in ascending order of the other index, exactly the reference's order.
                if (a.collide) {
                    const R2* envp = s_old + le * N;
                    if (env_nf) {
                        // rare: an env with a non-finite old position -- no cut-off (see env_cut2), every pair in
                        // ascending j, masses and sizes as in the loops below
                        const bool cached = a.cpos != nullptr;
                        const R2 pc = envp[i];
                        for (int j = 0; j < N; ++j) {
                            if (j == i) continue;
                            R2 q = envp[j];
                            T dx = (j < i) ? O::sub(q.x, pc.x) : O::sub(pc.x, q.x);   // delta = p_a - p_b, a<b
                            T dy = (j < i) ? O::sub(q.y, pc.y) : O::sub(pc.y, q.y);
                            const T dmin = HET ? O::add((j < i) ? s_het[N + j] : size_i, (j < i) ? size_i : s_het[N + j])
                                               : O::add(a.size, a.size);
                            T fx, fy;
                            contact_force<T>(dx, dy, dmin, a.margin, a.cforce, &fx, &fy, cached);
                            if (HET) {
                                T m_j = s_het[j];
                                if (j < i) { T c = -O::div((T)1, O::div(m_i, m_j)); Fx = O::add(O::mul(c, fx), Fx); Fy = O::add(O::mul(c, fy), Fy); }
                                else       { T r = O::div(m_j, m_i); Fx = O::add(O::mul(r, fx), Fx); Fy = O::add(O::mul(r, fy), Fy); }
                            } else {
                                if (j < i) { Fx = O::add(-fx, Fx); Fy = O::add(-fy, Fy); }
                                else       { Fx = O::add(fx, Fx);  Fy = O::add(fy, Fy); }
                            }
                        }
                    } else
                    if constexpr (FP) {
                        // candidate groups of four partners from the packed filter, then the reference's exact
                        // test and force for the members of flagged groups, in ascending j
                        const T dmin = O::add(a.size, a.size);                  // core.py:307
                        u64 near;
                        if (a.cells) {
                            // true near partners (exact cut-off test on the spot) from the 3 x 3 cells around me;
                            // an env with a far or non-finite agent falls back to testing every group
                            if (c_far[le]) near = (NP == 256) ? ~0ull : ((1ull << (NP >> 2)) - 1ull);
                            else near = cell_near_groups(c_head + le * CB, c_node + le * NP, a.cell_shift, cpos,
                                                         (float)p.x, (float)p.y, (float)a.cut2, i);
                        } else {
                            const float thr = ((float)a.cut2 - n_old) + filter_margin(n_old, __uint_as_float(s_nmax[le]));
                            near = filter_groups(reinterpret_cast<const ulonglong2*>(f_ro) + le * NG * 3, NG,
                                                 (float)p.x, (float)p.y, thr);
                        }
                        // Two phases keep the warp converged on the expensive part: (1) cheap exact cut-off test
                        // of the members of flagged groups, true near partners appended (ascending j) to a
                        // register list of up to 8 byte-sized indices; (2) the softplus force for the listed
                        // partners.  Dense clusters alternate between the phases.
                        u64 list = 0; int cnt = 0;
                        while (near | (u64)cnt) {
                            while (near && cnt <= 4) {
                                const int j4 = (__ffsll((long long)near) - 1) << 2;
                                near &= near - 1;
#pragma unroll
                                for (int jj = 0; jj < 4; ++jj) {
                                    const int j = j4 + jj;
                                    R2 q = envp[min(j, N - 1)];
                                    T dx = O::sub(p.x, q.x), dy = O::sub(p.y, q.y);
                                    T d2 = dx * dx + dy * dy;
                                    if (j < N && j != i && !(d2 >= a.cut2)) { list |= (u64)j << (8 * cnt); ++cnt; }
                                }
                            }
                            for (int k = 0; k < cnt; ++k) {
                                const int j = (int)(list >> (8 * k)) & 255;
                                R2 q = envp[j];
                                T dx = (j < i) ? O::sub(q.x, p.x) : O::sub(p.x, q.x);   // delta = p_a - p_b, a<b
                                T dy = (j < i) ? O::sub(q.y, p.y) : O::sub(p.y, q.y);
                                T fx, fy;
                                contact_force<T>(dx, dy, dmin, a.margin, a.cforce, &fx, &fy);
                                if (j < i) { Fx = O::add(-fx, Fx); Fy = O::add(-fy, Fy); }   // equal masses: ratio 1
                                else       { Fx = O::add(fx, Fx);  Fy = O::add(fy, Fy); }
                            }
                            list = 0; cnt = 0;
                        }
                    } else if (!HET) {
                        // uniform agents: per chunk of 32 partners, pass 1 builds a near-pair bitmask
                        // branch-free (7 instructions per pair), pass 2 evaluates the softplus force only
                        // for set bits, in ascending j (the reference's accumulation order).
                        const T dmin = O::add(a.size, a.size);                  // core.py:307
                        const bool cached = a.cpos != nullptr;                  // World.cache_dists (core.py:298-301)
                        const R2 p = envp[i];                                   // my position the contacts see (== p unless cached)
                        for (int j0 = 0; j0 < N; j0 += 32) {
                            const int jn = min(32, N - j0);
                            unsigned near = 0;
#pragma unroll 8
                            for (int jj = 0; jj < jn; ++jj) {
                                R2 q = envp[j0 + jj];
                                T dx = O::sub(p.x, q.x), dy = O::sub(p.y, q.y);
                                T d2 = dx * dx + dy * dy;
                                // Far pairs: softplus(-(d-dmin)/k) < exp(-kcut) -- below the rounding of
                                // F (DESIGN.md "contact cut-off").  !(>=) keeps NaN pairs; inf ones: env_nf above.
                                near |= (!(d2 >= a.cut2)) ? (1u << jj) : 0u;
                            }
                            if ((unsigned)(i - j0) < 32u) near &= ~(1u << (i - j0));
                            while (near) {
                                const int j = j0 + __ffs(near) - 1;
                                near &= near - 1;
                                R2 q = envp[j];
                                T dx = (j < i) ? O::sub(q.x, p.x) : O::sub(p.x, q.x);   // delta = p_a - p_b, a<b
                                T dy = (j < i) ? O::sub(q.y, p.y) : O::sub(p.y, q.y);
                                T fx, fy;
                                contact_force<T>(dx, dy, dmin, a.margin, a.cforce, &fx, &fy, cached);
                                if (j < i) { Fx = O::add(-fx, Fx); Fy = O::add(-fy, Fy); }   // equal masses: ratio 1
                                else       { Fx = O::add(fx, Fx);  Fy = O::add(fy, Fy); }
                            }
                        }
                    } else {
                        const bool cached = a.cpos != nullptr;
                        const R2 p = envp[i];                                   // my position the contacts see
                        for (int j = 0; j < N; ++j) {
                            if (j == i) continue;
                            R2 q = envp[j];
                            T dx = (j < i) ? O::sub(q.x, p.x) : O::sub(p.x, q.x);   // delta = p_a - p_b, a<b
                            T dy = (j < i) ? O::sub(q.y, p.y) : O::sub(p.y, q.y);
                            T d2 = dx * dx + dy * dy;
                            T dmin, cut2;
                            if (HET) {
                                dmin = O::add((j < i) ? s_het[N + j] : size_i, (j < i) ? size_i : s_het[N + j]);
                                T c = dmin + a.kcut * a.margin; cut2 = c * c;
                            } else {
                                dmin = O::add(a.size, a.size);                       // core.py:307
                                cut2 = a.cut2;
                            }
                            // Far pairs: softplus(-(d-dmin)/k) < exp(-kcut) -- below the rounding of F
                            // (DESIGN.md "contact cut-off").  !(>=) keeps NaN pairs; inf ones: env_nf above.
                            if (!(d2 >= cut2)) {
                                T fx, fy;
                                contact_force<T>(dx, dy, dmin, a.margin, a.cforce, &fx, &fy, cached);
                                if (HET) {
                                    T m_j = s_het[j];
                                    if (j < i) {       // i is entity b: force_b = -(1/ratio)*force, ratio = m_b/m_a
                                        T c = -O::div((T)1, O::div(m_i, m_j));
                                        Fx = O::add(O::mul(c, fx), Fx); Fy = O::add(O::mul(c, fy), Fy);
                                    } else {           // i is entity a: force_a = ratio*force
                                        T r = O::div(m_j, m_i);
                                        Fx = O::add(O::mul(r, fx), Fx); Fy = O::add(O::mul(r, fy), Fy);
                                    }
                                } else {               // equal masses: ratio == 1 exactly
                                    if (j < i) { Fx = O::add(-fx, Fx); Fy = O::add(-fy, Fy); }
                                    else       { Fx = O::add(fx, Fx);  Fy = O::add(fy, Fy); }
                                }
                            }
                        }
                    }
                }
                for (int w = 0; w < a.n_walls; ++w) {                          // core.py:255-261
                    T fx, fy;
                    wall_force<T>(a.walls[w], p.x, p.y, size_i, a.margin, a.cforce, &fx, &fy);
                    Fx = O::add(Fx, fx); Fy = O::add(Fy, fy);
                }
                // integrate_state (core.py:264-277)
                v.x = O::mul(v.x, a.keep); v.y = O::mul(v.y, a.keep);            // * (1 - damping)
                // F / m: exact without the division when every mass is 1
                const bool unit_mass = !HET && a.mass_one;
                v.x = O::add(v.x, O::mul(unit_mass ? Fx : O::div(Fx, m_i), a.dt));
                v.y = O::add(v.y, O::mul(unit_mass ? Fy : O::div(Fy, m_i), a.dt));
                T vmax = HET ? s_het[4 * N + i] : (a.has_vmax ? a.vmax : (T)-1);
                if (vmax >= (T)0) {
                    T sp = O::sqrt_(O::sq2(v.x, v.y));
                    if (sp > vmax) {
                        v.x = O::mul(O::div(v.x, sp), vmax);
                        v.y = O::mul(O::div(v.y, sp), vmax);
                    }
                }
                p.x = O::add(p.x, O::mul(v.x, a.dt));
                p.y = O::add(p.y, O::mul(v.y, a.dt));
                // update_agent_state (core.py:279-286)
                R2 c = O::make((T)0, (T)0);
                if (!a.silent) {
                    c = uc;
                    if (a.c_noise > (T)0) {
                        U4 r = philox(a.seed, ge, (uint32_t)i, tick0 + (uint32_t)ts, kCNoise);
                        T n0, n1; normal_pair<T>(r.x, r.y, &n0, &n1);
                        c.x = O::add(c.x, O::mul(n0, a.c_noise));
                        c.y = O::add(c.y, O::mul(n1, a.c_noise));
                    }
                }
                s_new[t] = p; s_v[t] = v; s_c[t] = c;
                if (!OBSREW || ts == a.n_steps - 1) {
                    a.pos[g] = p; a.vel[g] = v;
                    if (a.comm) a.comm[g] = c;
                }
            }
            if (!OBSREW) { tick_arrive(a.tick_dev, gridDim.x, a.n_steps, t == 0); return; }
            __syncthreads();
        }
        if constexpr (OM == 2 && sizeof(R2) == 8) {
            if (early && a.row_chunk) {
                rows_chunked();                                              // drains under the reward pass
            } else
            if (early) {
                // Dynamic 1/3 of every row, one warp per row, BEFORE the reward pass so that the stores drain
                // under it.  Pieces are 16-byte aligned on both ends: an even row sends [p_vel | other_pos | first
                // comm zero] (N+1 items) from its start; an odd row starts 8 bytes early with the previous
                // row's ideal_vel.  Only the first row of the tile (if odd) and the last (if even) need one
                // plain 8-byte store.
                R2* dyn2 = s_rt_dyn + wp_ * NB * rt_dyn;                         // NB staging buffers per warp
                const int nrows = nvalid * N;
                uint64_t pol;
                asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
                int pending = 0;
                // per-row bookkeeping hoisted out of the loop (it was ~200 of the ~250 warp instructions per row and
                // makes mid-size N issue-bound): a warp's rows are 8 apart, so they all have the SAME 16-byte phase;
                // (env, agent) of the row and its output pointer advance incrementally (N >= 48 > 8: one wrap at most)
                const bool odd = ((((size_t)tile0 * N) + (size_t)wp_) & 1) != 0;
                int rle = 0, ri = wp_;
                R2* out = a.obs + ((size_t)tile0 * N + wp_) * a.IPR;
                const size_t ostride = (size_t)(kBlock / 32) * a.IPR;
                for (int row = wp_; row < nrows; row += kBlock / 32, out += ostride, ri += kBlock / 32) {
                    if (ri >= N) { ri -= N; ++rle; }
                    R2* img = dyn2 + (NB == 2 ? (pending & 1) : 0) * rt_dyn;
                    if (lane_ == 0) {            // the buffer being refilled must have been read by its bulk copy
                        if (NB == 2) { if (pending >= 2) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
                        else if (pending >= 1) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                    }
                    __syncwarp();
                    const R2* P = s_new + rle * N;
                    const R2 pi = P[ri];
                    // layout of the staged piece: even [v, rel(N-1), 0]; odd (row > 0) [iv_prev, v, rel(N-1)];
                    // odd first row of the tile: [rel(N-1)] (p_vel goes out as a plain store)
                    const int off = odd ? (row > 0 ? 2 : 0) : 1;
                    for (int k = lane_; k < N - 1; k += 32) {                    // other_pos (formation_hd_env.py:55)
                        R2 pj = P[k + (k >= ri)];
                        img[off + k] = O::make(O::sub(pj.x, pi.x), O::sub(pj.y, pi.y));
                    }
                    if (lane_ == 0) {
                        if (!odd) { img[0] = s_v[row]; img[N] = FINOBS ? s_c[rle * N + (ri == 0)] : O::make((T)0, (T)0); }
                        else if (row > 0) { img[0] = s_iv[ri == 0 ? rle - 1 : rle]; img[1] = s_v[row]; }   // previous row's env
                        else O::stcs(out, s_v[row]);
                        if (!odd && row == nrows - 1) O::stcs(out + 3 * N - 1, s_iv[rle]);   // nobody follows
                    }
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    __syncwarp();
                    if (lane_ == 0) {
                        R2* dst = odd ? (row > 0 ? out - 1 : out + 1) : out;
                        const uint32_t bytes = (uint32_t)(((odd && row == 0) ? N - 1 : N + 1) * sizeof(R2));
                        asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;"
                                     :: "l"(dst), "r"(smem_u32(img)), "r"(bytes), "l"(pol) : "memory");
                        // static 2/3 from the env's shared image: even row items 1 .. 2N-2 (item 0 rode with the
                        // dynamic piece, item 2N-1 rides with the next row), odd row all 2N items
                        const R2* im0 = s_rt_img + (size_t)rle * 2 * rt_img;
                        R2* sdst = odd ? out + N : out + N + 1;
                        const R2* ssrc = odd ? im0 : im0 + rt_img + 1;
                        const uint32_t sbytes = (uint32_t)((odd ? 2 * N : 2 * N - 2) * sizeof(R2));
                        asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;"
                                     :: "l"(sdst), "r"(smem_u32(ssrc)), "r"(sbytes), "l"(pol) : "memory");
                        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                    }
                    ++pending;
                }
            }
        }

        // ================= Scenario.reward partials on the NEW state (Q16) ======================
        int col = 0;
        T mvx = 0, mvy = 0;
        float fcx = 0.f, fcy = 0.f, fnc = 0.f;                                // FP: my centred position, its norm^2
        if (SCN >= kScnPartial) {
            // formation_hd_partial_env.py:70-75: u - mean(u), v - mean(v) (agents / landmarks), summed in order
            if (active && (!(fabs(p.x) < (T)INFINITY) || !(fabs(p.y) < (T)INFINITY))) s_bad[le] = 1;
            if (t < 2 * nvalid) {
                const int qe = t >> 1;
                const int cnt = (t & 1) ? L : N;
                const R2* src = (t & 1) ? (s_s + qe * L) : (s_new + qe * N);
                T sx = 0, sy = 0;
                for (int j = 0; j < cnt; ++j) { R2 q = src[j]; sx = O::add(sx, q.x); sy = O::add(sy, q.y); }
                s_mean[t] = O::make(O::div(sx, (T)cnt), O::div(sy, (T)cnt));
            }
            __syncthreads();
            if (active) {
                const R2 mp = s_mean[2 * le];
                s_cen[t] = O::make(O::sub(p.x, mp.x), O::sub(p.y, mp.y));
            }
            __syncthreads();
        }
        if (SCN == kScnHD) {
            // a non-finite position makes the centroid, hence the whole shape term, NaN (Q9)
            if (active && (!(fabs(p.x) < (T)INFINITY) || !(fabs(p.y) < (T)INFINITY))) s_bad[le] = 1;
            if constexpr (FP) {
                if (a.cells && a.collide && active)                          // cell list of the NEW positions
                    cpos = cell_insert((float)p.x, (float)p.y, a.cell_inv_new, a.cell_shift, c_head + (EPC + le) * CB,
                                       c_node + (EPC + le) * NP, i, &c_far[EPC + le]);
                // centroid and mean velocity (formation_hd_env.py:65,68): butterfly sums over the lanes of
                // each env in the warp, one partial per (env, warp), combined in warp order after the barrier
                if (PHYS && t < EPC) s_nmax[t] = 0u;                         // re-arm for the next rollout step
                if (EPC > 1) {
                    // several envs per CTA: an env's lanes are cut by the warp boundaries at places that depend on
                    // its position in the tile, so butterfly partials would make the rounding of the sums -- and
                    // with it the results -- depend on how envs are sharded over launches / GPUs.  One thread per
                    // (env, quantity) sums in agent order instead (as the scalar path does).
                    if (t < 2 * nvalid) {
                        const int qe = t >> 1;
                        const R2* src = (t & 1) ? (s_v + qe * N) : (s_new + qe * N);
                        float sx = 0.f, sy = 0.f;
#pragma unroll 4
                        for (int j = 0; j < N; ++j) { R2 q = src[j]; sx += (float)q.x; sy += (float)q.y; }
                        f_part[(qe * 8) * 4 + 2 * (t & 1)] = sx;
                        f_part[(qe * 8) * 4 + 2 * (t & 1) + 1] = sy;
                    }
                } else {
                float a0 = inA ? (float)p.x : 0.f, a1 = inA ? (float)p.y : 0.f;
                float a2 = inA ? (float)v.x : 0.f, a3 = inA ? (float)v.y : 0.f;
#pragma unroll
                for (int off = 16; off; off >>= 1) {
                    a0 += __shfl_xor_sync(0xffffffffu, a0, off); a1 += __shfl_xor_sync(0xffffffffu, a1, off);
                    a2 += __shfl_xor_sync(0xffffffffu, a2, off); a3 += __shfl_xor_sync(0xffffffffu, a3, off);
                }
                if (maskA && lane_ == 0)
                    *reinterpret_cast<float4*>(f_part + (leA * 8 + wp_) * 4) = make_float4(a0, a1, a2, a3);
                if (maskB) {                                                 // warp-uniform
                    a0 = inB ? (float)p.x : 0.f; a1 = inB ? (float)p.y : 0.f;
                    a2 = inB ? (float)v.x : 0.f; a3 = inB ? (float)v.y : 0.f;
#pragma unroll
                    for (int off = 16; off; off >>= 1) {
                        a0 += __shfl_xor_sync(0xffffffffu, a0, off); a1 += __shfl_xor_sync(0xffffffffu, a1, off);
                        a2 += __shfl_xor_sync(0xffffffffu, a2, off); a3 += __shfl_xor_sync(0xffffffffu, a3, off);
                    }
                    if (lane_ == 0)
                        *reinterpret_cast<float4*>(f_part + ((leA + 1) * 8 + wp_) * 4) = make_float4(a0, a1, a2, a3);
                }
                }
            } else if (t < 2 * nvalid) {
                const int qe = t >> 1;
                const R2* src = (t & 1) ? (s_v + qe * N) : (s_new + qe * N);
                T sx = 0, sy = 0;
#pragma unroll 4
                for (int j = 0; j < N; ++j) { R2 q = src[j]; sx = O::add(sx, q.x); sy = O::add(sy, q.y); }
                s_mean[t] = O::make(O::div_count(sx, N), O::div_count(sy, N));   // np.mean: fp64 divides, fp32 multiplies by 1/N
            }
            __syncthreads();
            if constexpr (FP) {
                float sx = 0.f, sy = 0.f, svx = 0.f, svy = 0.f;
                if (active) {
#pragma unroll
                    for (int w = 0; w < kBlock / 32; ++w) {
                        const float4 q = *reinterpret_cast<const float4*>(f_part + (le * 8 + w) * 4);
                        sx += q.x; sy += q.y; svx += q.z; svy += q.w;
                    }
                }
                const float invN = 1.0f / (float)N;
                mvx = svx * invN; mvy = svy * invN;
                fcx = (float)p.x - sx * invN; fcy = (float)p.y - sy * invN;           // centred agent shape
                fnc = fcx * fcx + fcy * fcy;
                if (active) { RN(le, i, 0) = fcx; RN(le, i, 1) = fcy; RN(le, i, 2) = fnc; }
                env_atomic_max(s_nmax + EPC, __float_as_uint(fnc));
            } else if (active) {
                const R2 mp = s_mean[2 * le], mv = s_mean[2 * le + 1];
                mvx = mv.x; mvy = mv.y;
                s_cen[t] = O::make(O::sub(p.x, mp.x), O::sub(p.y, mp.y));      // centred agent shape
            }
            __syncthreads();
        }
        if constexpr (FP) {
            // collision candidates + both Hausdorff minima in one packed pass over the env (fg_pairs.cuh);
            // flagged groups get the reference's exact test (formation_hd_env.py:119-121; Q18), self excluded
            unsigned hbits = 0u;
            if (active) {
                const R2* envp = s_new + le * N;
                const R2 Si = s_s[t];
                const float thr = ((float)a.rthr2_hi - fnc) + filter_margin(fnc, __uint_as_float(s_nmax[EPC + le]));
                float rowmin, colmin;
                const ulonglong2* rn = reinterpret_cast<const ulonglong2*>(f_rn) + le * NG * 5;
                u64 hit = (a.collide && !a.cells)
                    ? reward_pass<true>(rn, NG, fcx, fcy, (float)Si.x, (float)Si.y, thr, &rowmin, &colmin)
                    : reward_pass<false>(rn, NG, fcx, fcy, (float)Si.x, (float)Si.y, thr, &rowmin, &colmin);
                if (a.cells && a.collide) {
                    // reward collisions (formation_hd_env.py:71-74,119-121; Q18) straight from the cell list of the
                    // new positions: a count, so the visiting order does not matter
                    if (c_far[EPC + le]) {
                        for (int j = 0; j < N; ++j) {
                            R2 q = envp[j];
                            const T dx = O::sub(q.x, p.x), dy = O::sub(q.y, p.y);
                            if (j != i && dx * dx + dy * dy < a.rthr2_hi) { if (O::norm2(dx, dy) < a.rthr) ++col; }
                        }
                    } else {
                        col = cell_count_collisions(c_head + (EPC + le) * CB, c_node + (EPC + le) * NP,
                                                    a.cell_shift, a.cell_inv_new, cpos, (float)p.x, (float)p.y,
                                                    (float)a.rthr2_hi, (float)a.rthr, i);
                    }
                }
                while (hit) {
                    const int j4 = (__ffsll((long long)hit) - 1) << 2;
                    hit &= hit - 1;
#pragma unroll
                    for (int jj = 0; jj < 4; ++jj) {
                        const int j = j4 + jj;
                        if (j >= N || j == i) continue;
                        R2 q = envp[j];
                        const T dx = O::sub(q.x, p.x), dy = O::sub(q.y, p.y);
                        // the thread's own group is always flagged: guarded squared test first, the
                        // reference's sqrt-then-compare (Q18) only for true candidates
                        if (dx * dx + dy * dy < a.rthr2_hi) { if (O::norm2(dx, dy) < a.rthr) ++col; }
                    }
                }
                hbits =__float_as_uint(fmaxf(rowmin, colmin));               // d2 >= 0: bit order == value order
            }
            env_atomic_max(reinterpret_cast<unsigned*>(s_rowmax), hbits);
            env_atomic_add(s_col, col);
        } else if (active) {
            const R2* envp = s_new + le * N;
            // is_collision: hd excludes self, threshold (s1+s2)/2 (formation_hd_env.py:73,119-121);
            // basic includes self, threshold s1+s2 (basic_formation_env.py:48-51,89-91)
            if (a.collide) {
                if (!HET) {
                    // candidates by squared distance (bitmask per 32 partners), exact sqrt test after (Q18)
                    for (int j0 = 0; j0 < N; j0 += 32) {
                        const int jn = min(32, N - j0);
                        unsigned hit = 0;
#pragma unroll 8
                        for (int jj = 0; jj < jn; ++jj) {
                            R2 q = envp[j0 + jj];
                            T dx = O::sub(q.x, p.x), dy = O::sub(q.y, p.y);
                            T d2 = dx * dx + dy * dy;
                            hit |= (d2 < a.rthr2_hi) ? (1u << jj) : 0u;
                        }
                        if (SCN != kScnBasic && (unsigned)(i - j0) < 32u) hit &= ~(1u << (i - j0));
                        while (hit) {
                            const int j = j0 + __ffs(hit) - 1;
                            hit &= hit - 1;
                            R2 q = envp[j];
                            if (O::norm2(O::sub(q.x, p.x), O::sub(q.y, p.y)) < a.rthr) ++col;
                        }
                    }
                } else {
                    const T size_i = s_het[N + i];
                    for (int j = 0; j < N; ++j) {
                        if (SCN != kScnBasic && j == i) continue;
                        R2 q = envp[j];
                        T dx = O::sub(q.x, p.x), dy = O::sub(q.y, p.y);
                        T d2 = dx * dx + dy * dy;
                        T thr = O::add(s_het[N + j], size_i);
                        if (SCN == kScnHD) thr = O::div(thr, (T)2);
                        if (d2 < thr * thr * (T)1.0001) { if (O::norm2(dx, dy) < thr) ++col; }
                    }
                }
            }
            if (SCN == kScnHD) {
                // reward part 1 (formation_hd_env.py:64-66): symmetric Hausdorff distance between the
                // centred agent shape C and the ideal shape S.  Thread i owns row i (min_j |C_i-S_j|^2)
                // and column i (min_j |C_j-S_i|^2); env-wide max via shared atomicMax on the bits.
                const R2* envs = s_s + le * N;
                const R2* envc = s_cen + le * N;
                const R2 Si = envs[i], Ci = envc[i];
                T rowmin = (T)INFINITY, colmin = (T)INFINITY;
#pragma unroll 4
                for (int j = 0; j < N; ++j) {
                    R2 Cj = envc[j]; R2 Sj = envs[j];
                    rowmin = fmin(rowmin, O::sq2(O::sub(Ci.x, Sj.x), O::sub(Ci.y, Sj.y)));
                    colmin = fmin(colmin, O::sq2(O::sub(Cj.x, Si.x), O::sub(Cj.y, Si.y)));
                }
                atomicMax(&s_rowmax[le], O::bits(fmax(rowmin, colmin)));   // d2 >= 0: bit order == value order
            }
            if (SCN >= kScnPartial) {
                // rows of the symmetric Hausdorff distance (formation_hd_partial_env.py:75): agent i against the
                // centred landmarks
                const R2 Ci = s_cen[t], ml = s_mean[2 * le + 1];
                const R2* envl = s_s + le * L;
                T rowmin = (T)INFINITY;
                for (int k = 0; k < L; ++k) {
                    R2 l = envl[k];
                    rowmin = fmin(rowmin, O::sq2(O::sub(Ci.x, O::sub(l.x, ml.x)), O::sub(Ci.y, O::sub(l.y, ml.y))));
                }
                atomicMax(&s_rowmax[le], O::bits(rowmin));
            }
            if (col) atomicAdd(&s_col[le], col);
        }
        if (SCN >= kScnPartial) {
            // columns: centred landmark k against all centred agents (one thread per (env, landmark))
            for (int q = t; q < nvalid * L; q += kBlock) {
                const int qe = (int)fastdiv((uint32_t)q, a.magic_l);
                const R2 ml = s_mean[2 * qe + 1];
                const R2 l = s_s[q];
                const R2 V = O::make(O::sub(l.x, ml.x), O::sub(l.y, ml.y));
                const R2* envc = s_cen + qe * N;
                T colmin = (T)INFINITY;
                for (int j = 0; j < N; ++j) {
                    R2 Cj = envc[j];
                    colmin = fmin(colmin, O::sq2(O::sub(Cj.x, V.x), O::sub(Cj.y, V.y)));
                }
                atomicMax(&s_rowmax[qe], O::bits(colmin));
            }
        }
        if (SCN == kScnBasic) {
            if (a.nan_flag && active && (!(fabs(p.x) < (T)INFINITY) || !(fabs(p.y) < (T)INFINITY))) s_bad[le] = 1;
            // reward part 1 (basic_formation_env.py:45-47): min over agents of |p_a - l_k| per landmark
            for (int q = t; q < nvalid * L; q += kBlock) {
                int qe = (int)fastdiv((uint32_t)q, a.magic_l);
                R2 l = s_s[q];
                const R2* envp = s_new + qe * N;
                T m = (T)INFINITY;
                bool nan_seen = false;
                for (int j = 0; j < N; ++j) {
                    R2 pj = envp[j];
                    T d = O::norm2sq(O::sub(pj.x, l.x), O::sub(pj.y, l.y));     // one sqrt after the loop (monotonic)
                    nan_seen |= (d != d);
                    m = fmin(m, d);
                }
                s_lmin[q] = nan_seen ? O::from_bits(~(Bits)0 >> 1) : O::sqrt_(m);
            }
        }
        __syncthreads();

        // ============ rewards, done, statistics (environment.py:126-138,172-177) ================
        stp += 1;                                                             // environment.py:114
        const bool dn = active && a.step && (stp >= a.world_length);
        if (active && i == 0) s_dn[le] = dn ? 1 : 0;
        if (active) {
            T base;
            if (SCN == kScnHD) {
                T form = -O::sqrt_(O::from_bits(s_rowmax[le]));                 // -max(dH, dH')
                if (s_bad[le]) form = O::from_bits(~(Bits)0 >> 1);              // NaN, as the reference
                T velr = O::norm2(O::sub(s_iv[le].x, mvx), O::sub(s_iv[le].y, mvy));   // :68-69
                base = O::sub(form, velr);
            } else if (SCN >= kScnPartial) {
                base = -O::sqrt_(O::from_bits(s_rowmax[le]));                   // no velocity term (:75)
                if (s_bad[le]) base = O::from_bits(~(Bits)0 >> 1);
            } else {
                base = (T)0;
                for (int k = 0; k < L; ++k) base = O::sub(base, s_lmin[le * L + k]);
            }
            T r = base;
            for (int c = 0; c < col; ++c) r = O::sub(r, (T)1);                 // rew -= 1 per collision
            const int coltot = s_col[le];
            // shared reward = sum_i r_i (environment.py:136): N*base - total collisions, in fp64
            const double R = (double)N * (double)base - (double)coltot;
            if (!FINOBS) a.reward[g] = (T)R;
            if (a.indiv) a.indiv[g] = r;
            if (a.done) a.done[g] = (uint8_t)(a.step ? (stp >= a.world_length) : 0);
            if (i == 0 && a.nan_flag && s_bad[le]) a.nan_flag[e] = 1;           // the reference's failure mode (Q9), sticky
            if (i == 0 && a.step) {
                T ret = (T)R;
                if (a.ep_return) { ret = a.ep_return[e] + (T)R; a.ep_return[e] = (dn && a.auto_reset) ? (T)0 : ret; }
                int ec = coltot;
                if (a.ep_coll) { ec += a.ep_coll[e]; a.ep_coll[e] = (dn && a.auto_reset) ? 0 : ec; }
                if (dn && a.stats) {             // per-CTA accumulators; one set of global atomics per CTA below
                    atomicAdd(&s_stat[0], 1.0);
                    atomicAdd(&s_stat[1], (double)ret);
                    atomicAdd(&s_stat[2], (double)ret * (double)ret);
                    atomicAdd(&s_stat[3], (double)ec);
                }
            }
        }

        // ======== VecEnv auto-reset (env_wrappers.py:14-18; reset_world formation_hd_env.py:77-95)
        if (PHYS && a.auto_reset) {
            if (__syncthreads_or(dn ? 1 : 0)) {
                const uint32_t tk = tick0 + (uint32_t)ts;
                R2 lraw = O::make((T)0, (T)0);
                if (dn) {
                    if constexpr (EXT) {                      // terminal block: the post-step state, before the reset
                        if (a.fin_pos) {
                            a.fin_pos[g] = p; a.fin_vel[g] = v;
                            if (!a.silent) a.fin_comm[g] = s_c[t];
                            if (SCN == kScnHD) {
                                a.fin_shape[g] = s_s[t];
                                if (i == 0) a.fin_ivel[e] = s_iv[le];
                            }
                        }
                    }
                    U4 r = philox(a.seed, ge, (uint32_t)i, tk, kResetAgent);
                    p = O::make(uniform_pm1<T>(r.x), uniform_pm1<T>(r.y));
                    v = O::make((T)0, (T)0);
                    s_new[t] = p; s_v[t] = v; s_c[t] = v;
                    if (SCN == kScnHD) {
                        U4 q = philox(a.seed, ge, (uint32_t)i, tk, kResetLandmark);
                        lraw = O::make(uniform_pm1<T>(q.x), uniform_pm1<T>(q.y));
                        uint32_t kt = 0;
                        if constexpr (EXT) {                  // target bank: the task's raw shape
                            if (a.tgt_count > 0) {
                                kt = target_task<T>(a, e, ge, tk);
                                lraw = a.tgt_shape[(size_t)kt * N + i];
                            }
                        }
                        s_old[t] = lraw;                      // scratch: s_old is dead after the physics
                        if (a.lm) a.lm[g] = lraw;
                        if (i == 0) {
                            U4 w = philox(a.seed, ge, 0u, tk, kResetIdealVel);
                            R2 iv = O::make(uniform_pm1<T>(w.x), uniform_pm1<T>(w.y));
                            if (EXT && a.tgt_count > 0 && a.tgt_vel) iv = a.tgt_vel[kt];
                            s_iv[le] = iv; a.ivel[e] = iv;
                        }
                    }
                    stp = 0;
                }
                if (SCN != kScnHD) {
                    for (int q = t; q < nvalid * L; q += kBlock) {
                        int qe = (int)fastdiv((uint32_t)q, a.magic_l), k = q - qe * L;
                        if (s_dn[qe]) {
                            if (EXT && a.fin_pos) a.fin_lm[(size_t)tile0 * L + q] = s_s[q];   // terminal block
                            U4 r = philox(a.seed, a.env_offset + (uint32_t)(tile0 + qe), (uint32_t)k, tk, kResetLandmark);
                            R2 l = O::make(uniform_pm1<T>(r.x), uniform_pm1<T>(r.y));
                            s_s[q] = l; a.lm[(size_t)tile0 * L + q] = l;
                        }
                    }
                }
                __syncthreads();
                if (dn && SCN == kScnHD) {
                    const R2* raw = s_old + le * N;
                    T sx = 0, sy = 0;
                    for (int j = 0; j < N; ++j) { sx = O::add(sx, raw[j].x); sy = O::add(sy, raw[j].y); }
                    R2 S = O::make(O::sub(lraw.x, O::div(sx, (T)N)), O::sub(lraw.y, O::div(sy, (T)N)));  // :93
                    s_s[t] = S; a.shape[g] = S;
                    if constexpr (FP) { RN(le, i, 3) = (float)S.x; RN(le, i, 4) = (float)S.y; }
                }
                if (dn && ts == a.n_steps - 1) { a.pos[g] = p; a.vel[g] = v; if (a.comm) a.comm[g] = v; }
                __syncthreads();
            }
        }
        if (active && i == 0 && a.step) a.step[e] = stp;

        // hd observation side effect (formation_hd_env.py:40-44): every landmark moves by
        // mean(agent pos) - mean(landmark pos).  Visualisation only; skipped when lm == NULL.
        if (SCN == kScnHD && a.lm) {
            R2 l = O::make((T)0, (T)0);
            if (active) { l = a.lm[g]; s_old[t] = l; }       // s_old is scratch after the physics
            __syncthreads();
            if (active) {
                const R2* envp = s_new + le * N;
                const R2* envl = s_old + le * N;
                T sx = 0, sy = 0, lx = 0, ly = 0;
                for (int j = 0; j < N; ++j) {
                    sx = O::add(sx, envp[j].x); sy = O::add(sy, envp[j].y);
                    lx = O::add(lx, envl[j].x); ly = O::add(ly, envl[j].y);
                }
                T ddx = O::sub(O::div(sx, (T)N), O::div(lx, (T)N));
                T ddy = O::sub(O::div(sy, (T)N), O::div(ly, (T)N));
                a.lm[g] = O::make(O::add(l.x, ddx), O::add(l.y, ddy));
            }
            __syncthreads();
        }

        // ================= observation rows (formation_hd_env.py:52-59 / basic :29-41) ==========
        // The tile's rows form ONE contiguous span of nvalid*N*IPR R2 items in HBM; consecutive
        // threads write consecutive items (8 B fp32 / 16 B fp64 each): fully coalesced stores.
        if (early) {
            // the shared images / staging buffers must outlive the bulk copies' reads (kernel exit, or the next
            // rollout step that restages them)
            if (lane_ == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
            __syncwarp();
        } else if (a.obs) {
            const int IPR = a.IPR;
            if (OM == 2 && a.row_chunk) {
                __syncthreads();                                                 // (reset) state of every env is in place
                rows_chunked();
                if (t == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                __syncthreads();
            } else if (OM == 2) {
                // Long hd rows, silent agents: 2/3 of every row ([comm zeros | ideal_shape | ideal_vel]) is the
                // same for all rows of an env, so it is built ONCE per env in shared memory (in both
                // 16-byte phases) and bulk-stored N times from there; only the N dynamic items of a row
                // are staged per row.  Per row: ~6 instructions per dynamic item + 2 bulk stores.
                const int lane = t & 31, wp = t >> 5;
                for (int qe = 0; qe < nvalid; ++qe) {
                    R2* im0 = s_rt_img + (size_t)qe * 2 * rt_img;
                    R2* im1 = im0 + rt_img;
                    for (int k = t; k < 2 * N; k += kBlock) {
                        // (comm zeros of silent agents; fg_obs_gather takes them from s_c: NaN for a slot without a record)
                        R2 val = (k < N - 1) ? (FINOBS ? s_c[qe * N + k] : O::make((T)0, (T)0))
                                             : (k < 2 * N - 1 ? s_s[qe * N + (k - (N - 1))] : s_iv[qe]);
                        im0[k] = val; im1[k] = val;
                    }
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncthreads();
                R2* dyn2 = s_rt_dyn + wp * NB * rt_dyn;                          // NB staging buffers per warp
                const int nrows = nvalid * N;
                int pending = 0;
                for (int row = wp; row < nrows; row += kBlock / 32) {
                    R2* dyn = dyn2 + (NB == 2 ? (pending & 1) : 0) * rt_dyn;
                    const int rle = (int)fastdiv((uint32_t)row, a.magic_n);
                    const int ri = row - rle * N;
                    R2* out = a.obs + ((size_t)tile0 * N + row) * IPR;
                    const uint32_t ph = ((uint32_t)(uintptr_t)out & 15u) ? 1u : 0u;     // odd 8-byte slot (fp32 only)
                    R2* img = dyn + ph;                                                 // same phase as `out`
                    // the buffer being refilled was sent two rows ago: at most one younger group may be in flight
                    if (lane == 0) {
                        if (NB == 2) { if (pending >= 2) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
                        else if (pending >= 1) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                    }
                    __syncwarp();
                    const R2* P = s_new + rle * N;
                    const R2 pi = P[ri];
                    if (lane == 0) img[0] = s_v[row];                                   // p_vel
                    for (int k = lane; k < N - 1; k += 32) {                            // other_pos
                        R2 pj = P[k + (k >= ri)];
                        img[1 + k] = O::make(O::sub(pj.x, pi.x), O::sub(pj.y, pi.y));
                    }
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    __syncwarp();
                    row_piece_store<R2>(out, img, (uint32_t)(N * sizeof(R2)), lane);
                    // static part: starts N items later -> opposite phase when sizeof(R2) == 8 and N is odd
                    R2* outs = out + N;
                    const uint32_t phs = ((uint32_t)(uintptr_t)outs & 15u) ? 1u : 0u;
                    const R2* ims = s_rt_img + (size_t)rle * 2 * rt_img + (phs ? rt_img : 0);
                    // image phase: im0 is 16-byte aligned, im1 = im0 + (2N+1) items is 8 mod 16 (fp32)
                    row_piece_store<R2>(outs, ims, (uint32_t)(2 * N * sizeof(R2)), lane);
                    if (lane == 0) asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                    ++pending;
                }
                // the images must outlive the bulk copies' reads (kernel exit or the next rollout step)
                if (pending && lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                __syncthreads();
            } else if (OM == 3) {
                // Short rows: every thread stages ITS OWN row in shared memory with simple loops (no per-item
                // (row, item) decode); the tile's rows are ONE contiguous span of HBM, which leaves as one TMA
                // bulk store (16-byte aligned middle) plus at most one 8-byte head / tail item.
                R2* out = a.obs + (size_t)tile0 * N * IPR;
                R2* img = s_rt_img + (((uint32_t)(uintptr_t)out & 15u) ? 1 : 0);      // same 16-byte phase as `out`
                if (active) {
                    R2* row = img + (size_t)t * IPR;
                    const R2* P = s_new + le * N;
                    const R2* Cm = s_c + le * N;
                    row[0] = v;                                                        // p_vel
                    int base = 1;
                    if (SCN == kScnBasic) {
                        row[1] = p;                                                    // p_pos
                        const R2* Lm = s_s + le * L;
                        for (int k = 0; k < L; ++k) { R2 l = Lm[k]; row[2 + k] = O::make(O::sub(l.x, p.x), O::sub(l.y, p.y)); }
                        base = 2 + L;
                    } else if (SCN >= kScnPartial) {
                        const R2* Lm = s_s + le * L;
                        for (int k = 0; k < L; ++k) row[1 + k] = Lm[k];                // landmarks, absolute
                        base = 1 + L;
                    }
                    int nrel = N - 1;
                    if (SCN == kScnPartial) {                                          // agents i+1 .. i+num_obs, cyclic
                        nrel = a.num_obs;
                        int j = i;
                        for (int m = 0; m < nrel; ++m) {
                            j = (j + 1 == N) ? 0 : j + 1;
                            R2 pj = P[j];
                            row[base + m] = O::make(O::sub(pj.x, p.x), O::sub(pj.y, p.y));
                        }
                    } else {
                        for (int m = 0; m < N - 1; ++m) {                              // other_pos, j != i ascending
                            R2 pj = P[m + (m >= i)];
                            T dx = O::sub(pj.x, p.x), dy = O::sub(pj.y, p.y);
                            if (SCN == kScnRange) {                                    // np.clip keeps NaN
                                const T lo = -a.obs_range, hi = a.obs_range;
                                dx = (dx < lo) ? lo : ((dx > hi) ? hi : dx);
                                dy = (dy < lo) ? lo : ((dy > hi) ? hi : dy);
                            }
                            row[base + m] = O::make(dx, dy);
                        }
                    }
                    for (int m = 0; m < N - 1; ++m) row[base + nrel + m] = Cm[m + (m >= i)];   // comm of the others
                    if (SCN == kScnHD) {
                        const R2* Sh = s_s + le * N;
                        for (int k = 0; k < N; ++k) row[2 * N - 1 + k] = Sh[k];        // ideal_shape.flatten()
                        row[3 * N - 1] = s_iv[le];                                     // ideal_vel
                    }
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncthreads();
                if (t < 32) {
                    row_piece_store<R2>(out, img, (uint32_t)((size_t)nvalid * N * IPR * sizeof(R2)), t);
                    if (t == 0) {
                        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                        // the image must outlive the bulk copy's reads (kernel exit or the next rollout step)
                        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                    }
                }
                __syncthreads();
            } else if (OM == 1) {
                // Long rows (N >= 16): one warp per row, one simple loop per row segment -- no per-item
                // (row, item) decode; consecutive lanes store consecutive 8-byte items (256 B per
                // instruction, rows are contiguous in HBM).  st.global.cs: write-once streaming data.
                const int lane = t & 31;
                const int nrows = nvalid * N;
                for (int row = t >> 5; row < nrows; row += kBlock / 32) {
                    const int rle = (int)fastdiv((uint32_t)row, a.magic_n);
                    const int ri = row - rle * N;
                    R2* out = a.obs + ((size_t)tile0 * N + row) * IPR;
                    const R2* P = s_new + rle * N;
                    const R2 pi = P[ri];
                    if (lane == 0) O::stcs(out, s_v[row]);                              // p_vel
                    int base = 1;
                    if (SCN == kScnBasic) {
                        if (lane == 1) O::stcs(out + 1, pi);                            // p_pos
                        const R2* Lm = s_s + rle * L;
                        for (int k = lane; k < L; k += 32) {                            // landmarks - p
                            R2 l = Lm[k];
                            O::stcs(out + 2 + k, O::make(O::sub(l.x, pi.x), O::sub(l.y, pi.y)));
                        }
                        base = 2 + L;
                    }
                    for (int k = lane; k < N - 1; k += 32) {                            // other_pos
                        R2 pj = P[k + (k >= ri)];
                        O::stcs(out + base + k, O::make(O::sub(pj.x, pi.x), O::sub(pj.y, pi.y)));
                    }
                    const R2* Cm = s_c + rle * N;
                    for (int k = lane; k < N - 1; k += 32)                              // comm
                        O::stcs(out + base + (N - 1) + k, Cm[k + (k >= ri)]);
                    if (SCN == kScnHD) {
                        const R2* Sh = s_s + rle * N;
                        for (int k = lane; k < N; k += 32) O::stcs(out + 2 * N - 1 + k, Sh[k]);   // ideal_shape
                        if (lane == 0) O::stcs(out + 3 * N - 1, s_iv[rle]);             // ideal_vel
                    }
                }
            } else {
                const uint32_t total = (uint32_t)(nvalid * N * IPR);
                R2* out = a.obs + (size_t)tile0 * N * IPR;
                for (uint32_t q = t; q < total; q += kBlock) {
                    const uint32_t row = fastdiv(q, a.magic_ipr);          // (local env, agent) row
                    const int k = (int)(q - row * IPR);                    // item within the row
                    const int rle = (int)fastdiv(row, a.magic_n);
                    const int ri = (int)row - rle * N;
                    R2 val;
                    if (SCN == kScnHD) {
                        if (k == 0) val = s_v[row];                                        // p_vel
                        else if (k < N) {                                                  // other_pos
                            int j = k - 1; j += (j >= ri);
                            R2 pj = s_new[rle * N + j], pi = s_new[row];
                            val = O::make(O::sub(pj.x, pi.x), O::sub(pj.y, pi.y));
                        } else if (k < 2 * N - 1) {                                        // comm
                            int j = k - N; j += (j >= ri);
                            val = s_c[rle * N + j];
                        } else if (k < 3 * N - 1) val = s_s[rle * N + (k - (2 * N - 1))];  // ideal_shape
                        else val = s_iv[rle];                                              // ideal_vel
                    } else if (SCN >= kScnPartial) {
                        // [p_vel | landmark positions (absolute) | other_pos | comm of the others]
                        // (formation_hd_partial_env.py:42-66, formation_hd_partial_range_env.py:42-54)
                        const int nob = (SCN == kScnPartial) ? a.num_obs : N - 1;
                        if (k == 0) val = s_v[row];
                        else if (k < 1 + L) val = s_s[rle * L + (k - 1)];
                        else if (k < 1 + L + nob) {
                            const int m = k - (1 + L);
                            const R2 pi = s_new[row];
                            if (SCN == kScnPartial) {                      // agents i+1 .. i+num_obs, cyclic (:53-55)
                                int j = ri + 1 + m;
                                j -= (int)fastdiv((uint32_t)j, a.magic_n) * N;
                                R2 pj = s_new[rle * N + j];
                                val = O::make(O::sub(pj.x, pi.x), O::sub(pj.y, pi.y));
                            } else {                                       // all others, clipped to the range (:53)
                                const int j = m + (m >= ri);
                                R2 pj = s_new[rle * N + j];
                                T dx = O::sub(pj.x, pi.x), dy = O::sub(pj.y, pi.y);
                                const T lo = -a.obs_range, hi = a.obs_range;   // np.clip keeps NaN
                                dx = (dx < lo) ? lo : ((dx > hi) ? hi : dx);
                                dy = (dy < lo) ? lo : ((dy > hi) ? hi : dy);
                                val = O::make(dx, dy);
                            }
                        } else {
                            int j = k - (1 + L + nob); j += (j >= ri);
                            val = s_c[rle * N + j];
                        }
                    } else {
                        if (k == 0) val = s_v[row];                                        // p_vel
                        else if (k == 1) val = s_new[row];                                 // p_pos
                        else if (k < 2 + L) {                                              // landmarks - p
                            R2 l = s_s[rle * L + (k - 2)], pi = s_new[row];
                            val = O::make(O::sub(l.x, pi.x), O::sub(l.y, pi.y));
                        } else if (k < 2 + L + (N - 1)) {                                  // other_pos
                            int j = k - (2 + L); j += (j >= ri);
                            R2 pj = s_new[rle * N + j], pi = s_new[row];
                            val = O::make(O::sub(pj.x, pi.x), O::sub(pj.y, pi.y));
                        } else {                                                           // comm
                            int j = k - (2 + L + (N - 1)); j += (j >= ri);
                            val = s_c[rle * N + j];
                        }
                    }
                    out[q] = val;
                }
            }
        }

        if (!PHYS) break;
        // next step of an in-kernel rollout: the new positions become the old ones
        R2* tmp = s_old; s_old = s_new; s_new = tmp;
    }
    if (OBSREW && a.stats) {
        __syncthreads();
        if (t < 4 && s_stat[0] != 0.0) atomicAdd(&a.stats[t], s_stat[t]);
    }
    if (PHYS) tick_arrive(a.tick_dev, gridDim.x, a.n_steps, t == 0);
}

// ------------------------------------------------------------------------------------------------
// Scenario.reset_world + env.current_step = 0 for masked envs; one thread per env (reset of a whole
// batch is off the hot loop; in-episode resets happen inside k_step).  Same Philox counters and the
// same arithmetic as the in-kernel auto-reset, so both produce bit-identical states.
template <typename T, int SCN>
__global__ void k_reset(const __grid_constant__ KArgs<T> a, const uint8_t* __restrict__ mask) {
    typedef Ops<T> O;
    typedef typename O::R2 R2;
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= a.E) return;
    if (mask && !mask[e]) return;
    const int N = a.N, L = a.L;
    const uint32_t ge = a.env_offset + (uint32_t)e;
    const uint32_t tick0 = a.tick + (a.tick_dev ? a.tick_dev[0] : 0u);
    const R2 zero = O::make((T)0, (T)0);
    for (int i = 0; i < N; ++i) {
        U4 r = philox(a.seed, ge, (uint32_t)i, tick0, kResetAgent);
        size_t g = (size_t)e * N + i;
        a.pos[g] = O::make(uniform_pm1<T>(r.x), uniform_pm1<T>(r.y));
        a.vel[g] = zero;
        if (a.comm) a.comm[g] = zero;
    }
    // formation_hd_env with a target bank: the task's raw shape replaces the landmark draws (same centring below)
    uint32_t kt = 0;
    const R2* bank = nullptr;
    if (SCN == kScnHD && a.tgt_count > 0) {
        kt = target_task<T>(a, e, ge, tick0);
        bank = a.tgt_shape + (size_t)kt * N;
    }
    T sx = 0, sy = 0;
    for (int k = 0; k < L; ++k) {
        U4 r = philox(a.seed, ge, (uint32_t)k, tick0, kResetLandmark);
        R2 l = bank ? bank[k] : O::make(uniform_pm1<T>(r.x), uniform_pm1<T>(r.y));
        sx = O::add(sx, l.x); sy = O::add(sy, l.y);
        if (a.lm) a.lm[(size_t)e * L + k] = l;
    }
    if (SCN == kScnHD) {
        T mx = O::div(sx, (T)N), my = O::div(sy, (T)N);
        for (int k = 0; k < N; ++k) {
            U4 r = philox(a.seed, ge, (uint32_t)k, tick0, kResetLandmark);
            R2 l = bank ? bank[k] : O::make(uniform_pm1<T>(r.x), uniform_pm1<T>(r.y));
            a.shape[(size_t)e * N + k] = O::make(O::sub(l.x, mx), O::sub(l.y, my));
        }
        U4 w = philox(a.seed, ge, 0u, tick0, kResetIdealVel);
        a.ivel[e] = (bank && a.tgt_vel) ? a.tgt_vel[kt] : O::make(uniform_pm1<T>(w.x), uniform_pm1<T>(w.y));
    }
    if (a.step) a.step[e] = 0;
    if (a.ep_return) a.ep_return[e] = (T)0;
    if (a.ep_coll) a.ep_coll[e] = 0;
}

// Random policy act ~ U(-1,1) (test.py:20); same counters as the in-kernel rollout.  32-bit indices
// (E*N < 2^31 is checked by the ABI): one exact 32-bit division per thread, then (env, agent) advance
// incrementally along the grid-stride loop -- the kernel is a pure Philox + store stream (the 64-bit
// `g / N` per element it used to carry cost more than the ten Philox rounds).
template <typename T>
__global__ void __launch_bounds__(256) k_random_actions(typename Ops<T>::R2* __restrict__ act, uint32_t total, uint32_t N,
                                                        uint64_t seed, uint32_t tick, uint32_t env_offset,
                                                        const uint32_t* __restrict__ tick_dev) {
    if (tick_dev) tick += tick_dev[0];
    const uint32_t stride = gridDim.x * blockDim.x;
    const uint32_t se = stride / N, si = stride - se * N;
    uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t e = g / N, i = g - e * N;
    for (; g < total; g += stride) {
        U4 r = philox(seed, env_offset + e, i, tick, kAction);
        act[g] = Ops<T>::make(uniform_pm1<T>(r.x), uniform_pm1<T>(r.y));
        e += se; i += si;
        if (i >= N) { i -= N; ++e; }
    }
}

// World.calculate_distances (core.py:156-180) for every env: entity positions ent [E,M,2] (agents, then landmarks),
// sizes [M] -> vect [E,M,M,2] (p_a - p_b above the diagonal, its negative below, 0 on it), mag [E,M,M]
// (np.linalg.norm(axis=2): sqrt(x*x + y*y)), collisions [E,M,M] (mag <= min_dists; min_dists = size_a + size_b off
// the diagonal, 0 on it -> the diagonal is True, as in the reference), min_dists [M,M].
template <typename T>
__global__ void __launch_bounds__(256) k_pair_distances(const typename Ops<T>::R2* __restrict__ ent, const T* __restrict__ size,
                                                        int E, int M, typename Ops<T>::R2* __restrict__ vect,
                                                        T* __restrict__ mag, uint8_t* __restrict__ coll, T* __restrict__ mind) {
    typedef Ops<T> O;
    const size_t total = (size_t)E * M * M;
    for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < total; q += (size_t)gridDim.x * blockDim.x) {
        const int b = (int)(q % M), a_ = (int)((q / M) % M);
        const size_t e = q / ((size_t)M * M);
        const int lo = a_ < b ? a_ : b, hi = a_ < b ? b : a_;
        const typename O::R2 pl = ent[e * M + lo], ph = ent[e * M + hi];
        T dx = O::sub(pl.x, ph.x), dy = O::sub(pl.y, ph.y);                // delta_pos = p_ia - p_ib, ia < ib (:174)
        if (a_ == b) { dx = (T)0; dy = (T)0; }
        else if (a_ > b) { dx = -dx; dy = -dy; }                           // cached_dist_vect[ib, ia] = -delta_pos (:176)
        const T m = O::sqrt_(O::sq2(dx, dy));
        const T md = a_ == b ? (T)0 : O::add(size[lo], size[hi]);         // min_dists (:161-168)
        vect[q] = O::make(dx, dy);
        mag[q] = m;
        coll[q] = (uint8_t)(m <= md);                                      // :180
        if (e == 0) mind[(size_t)a_ * M + b] = md;
    }
}

}  // namespace fg
