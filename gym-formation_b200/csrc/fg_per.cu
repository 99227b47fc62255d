// fg_per.cu -- prioritized replay on the device (sm_100a): a 32-ary sum/min tree over the transitions of a
// state-record replay buffer, proportional sampling with importance weights, and priority updates.
//
// Tree (include/formation_gym_b200.h fg_per): level 0 is the M = slots*envs leaves (leaf j*E + e for slot j, env e),
// read as padded with zeros to a multiple of 32; node i of level k+1 reduces nodes 32i .. 32i+31 of level k (children
// past the end of a level read as sum 0 / min +inf).  Levels 1 .. depth are stored bottom level first in `sum` / `min`;
// the top level is the root.  A node's sum is the butterfly of its 32 children (v_l += v_{l^off}, off = 16 .. 1: one
// __shfl_xor reduction, taken from lane 0) and its min the minimum over the nonzero leaves below (+inf for none), so the
// tree is a pure function of the leaves: every writer recomputes a node from its finished children, level by level
// (one launch per level), and concurrent writers of one node store identical bits.  Nothing accumulates atomically.
//
// Kernels are warp-shaped: a warp owns one node (its 32 children are one coalesced 256-byte load) or one draw.
#include <stdint.h>
#include <cmath>

#include "fg_host.cuh"

namespace {

constexpr int kMaxDepth = 8;                                  // M <= 2^40 leaves: ceil(40 / 5) levels
constexpr long long kMaxLeaves = 1ll << 40;
constexpr unsigned kFull = 0xffffffffu;
constexpr int kThreads = 256;                                 // 8 warps per CTA

// Device view of an fg_per with its layout: cnt[k] nodes at level k (cnt[0] = M leaves), level k >= 1 stored at
// sum/min + off[k]; the root is sum/min[off[depth]].
struct Tree {
    double* leaf; double* sum; double* mn; double* max_leaf; int64_t* stamp; int64_t* prev; int* owner;
    long long T, E, M;
    int depth;
    long long cnt[kMaxDepth + 1], off[kMaxDepth + 1];
};

bool aligned(const void* p, size_t a) { return ((uintptr_t)p % a) == 0; }

// Layout of M leaves: levels until one node is left (M = 1 still has a root above its one leaf).
void layout(long long M, Tree* t, long long* nodes, int* depth) {
    long long n = M, total = 0;
    int d = 0;
    if (t) t->cnt[0] = M;
    do {
        n = (n + 31) / 32;
        ++d;
        if (t) { t->cnt[d] = n; t->off[d] = total; }
        total += n;
    } while (n > 1);
    *nodes = total;
    *depth = d;
}

int check_sizes(long long slots, long long envs, const char* who) {
    if (slots < 1 || envs < 1) return fail(FG_ERR_ARG, "%s: slots and envs must be >= 1", who);
    if (slots > kMaxLeaves / envs) return fail(FG_ERR_ARG, "%s: slots * envs must be <= 2^40", who);
    return FG_OK;
}

int make_tree(const fg_per* p, Tree* t, const char* who) {
    if (!p) return fail(FG_ERR_ARG, "%s: the tree must be non-null", who);
    int rc = check_sizes(p->slots, p->envs, who);
    if (rc) return rc;
    if (!p->leaf || !p->sum || !p->min || !p->max_leaf || !p->stamp || !p->prev || !p->scratch)
        return fail(FG_ERR_ARG, "%s: fg_per arrays must be non-null", who);
    if (!aligned(p->leaf, 8) || !aligned(p->sum, 8) || !aligned(p->min, 8) || !aligned(p->max_leaf, 8) ||
        !aligned(p->stamp, 8) || !aligned(p->prev, 8) || !aligned(p->scratch, 4))
        return fail(FG_ERR_ARG, "%s: fg_per arrays must be 8-byte aligned (scratch: 4-byte)", who);
    t->leaf = p->leaf; t->sum = p->sum; t->mn = p->min; t->max_leaf = p->max_leaf;
    t->stamp = p->stamp; t->prev = p->prev; t->owner = (int*)p->scratch;
    t->T = p->slots; t->E = p->envs; t->M = p->slots * p->envs;
    long long nodes;
    layout(t->M, t, &nodes, &t->depth);
    return FG_OK;
}

unsigned grid_for(long long threads, long long cap = 1ll << 30) {
    long long g = (threads + kThreads - 1) / kThreads;
    return (unsigned)(g < 1 ? 1 : (g > cap ? cap : g));
}

// ------------------------------------------------------------------ device side
__device__ __forceinline__ double child_sum(const Tree& t, int lvl, long long i) {
    if (i >= t.cnt[lvl]) return 0.0;
    return lvl == 0 ? t.leaf[i] : t.sum[t.off[lvl] + i];
}

// Node `node` of level k (>= 1) from its children at level k - 1; the whole warp calls it with the same node.
__device__ __forceinline__ void reduce_node(const Tree& t, int k, long long node, int lane) {
    const long long i = node * 32 + lane;
    double s = 0.0, m = INFINITY;
    if (i < t.cnt[k - 1]) {
        if (k == 1) { s = t.leaf[i]; if (s > 0.0) m = s; }
        else { s = t.sum[t.off[k - 1] + i]; m = t.mn[t.off[k - 1] + i]; }
    }
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) {
        s = s + __shfl_xor_sync(kFull, s, o);
        m = fmin(m, __shfl_xor_sync(kFull, m, o));
    }
    if (lane == 0) { t.sum[t.off[k] + node] = s; t.mn[t.off[k] + node] = m; }
}

// Level k of the tree: warp w recomputes node idx[w] >> 5k (idx: leaf indices, entries outside [0, M) skipped) when
// idx is given, else node lo0 + w for w < n0, then lo1 + (w - n0) for w < n0 + n1.  reset: owner[idx[w]] = 0 for
// w < n_reset (the update's duplicate resolution, done once the write kernel has finished reading it).
__global__ void __launch_bounds__(kThreads) k_per_level(Tree t, int k, const int64_t* __restrict__ idx, long long n_idx,
                                                        long long lo0, long long n0, long long lo1, long long n1,
                                                        const int64_t* __restrict__ reset, long long n_reset) {
    const int lane = threadIdx.x & 31;
    const long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (reset && w < n_reset && lane == 0) {
        const long long j = reset[w];
        if (j >= 0 && j < t.M) t.owner[j] = 0;
    }
    long long node = -1;
    if (idx) {
        if (w < n_idx) {
            const long long j = idx[w];
            if (j >= 0 && j < t.M) node = j >> (5 * k);
        }
    } else if (w < n0) {
        node = lo0 + w;
    } else if (w < n0 + n1) {
        node = lo1 + (w - n0);
    }
    if (node >= 0) reduce_node(t, k, node, lane);            // (warp-uniform)
}

// fg_per_fill, leaf part: leaves of `slot` := *max_leaf (valid) or 0, leaves of `drop` (>= 0) := 0; stamp / prev.
__global__ void __launch_bounds__(kThreads) k_per_fill(Tree t, long long slot, long long prev, long long stamp, int valid,
                                                       long long drop) {
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x, stride = (long long)gridDim.x * blockDim.x;
    const double v = valid ? *t.max_leaf : 0.0;
    for (long long e = tid; e < t.E; e += stride) {
        t.leaf[slot * t.E + e] = v;
        if (drop >= 0) t.leaf[drop * t.E + e] = 0.0;
    }
    if (tid == 0) { t.stamp[slot] = stamp; t.prev[slot] = prev; }
}

template <typename TD>
__device__ __forceinline__ bool per_applies(const Tree& t, long long j, int64_t st, TD td) {
    return j >= 0 && j < t.M && isfinite((double)td) && t.leaf[j] > 0.0 && t.stamp[j / t.E] == st;
}

// fg_per_update, step 1: every applicable entry offers its batch position; the largest wins (numpy a[idx] = v).
template <typename TD>
__global__ void __launch_bounds__(kThreads) k_per_claim(Tree t, const int64_t* __restrict__ idx,
                                                        const int64_t* __restrict__ st, const TD* __restrict__ td, int B) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const long long j = idx[b];
    if (per_applies(t, j, st[b], td[b])) atomicMax(&t.owner[j], b + 1);
}

// step 2: the winners write their leaves and raise max_leaf (positive doubles order like their bit patterns).  The
// warp's maximum goes out in ONE atomic: B same-address atomics would serialise at one L2 slice, and max is exact.
template <typename TD>
__global__ void __launch_bounds__(kThreads) k_per_write(Tree t, const int64_t* __restrict__ idx,
                                                        const TD* __restrict__ td, int B, double alpha, double eps) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long bits = 0;                             // 0: nothing written by this lane
    if (b < B) {
        const long long j = idx[b];
        if (j >= 0 && j < t.M && t.owner[j] == b + 1) {
            const double v = fmin(fmax(pow(fabs((double)td[b]) + eps, alpha), 0x1p-1022), 0x1p960);
            t.leaf[j] = v;
            bits = (unsigned long long)__double_as_longlong(v);
        }
    }
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) bits = max(bits, __shfl_xor_sync(kFull, bits, o));   // (full warps: 256-thread CTAs)
    if ((threadIdx.x & 31) == 0 && bits) atomicMax((unsigned long long*)t.max_leaf, bits);
}

// fg_per_sample: one warp per draw.  Descend from the root: at each node take the smallest child k with c_k > 0 and
// x < P_k (inclusive prefix sum), else the last child with c_k > 0, then x -= P_{k-1} clamped into [0, c_k).  A zero
// child is never taken, so a zero leaf is never returned.  The warp then writes the transition's record rows, done,
// importance weight (root.min / leaf)^beta and its actions / reward rows.
template <typename T>
__global__ void __launch_bounds__(kThreads) k_per_sample(Tree t, const double* __restrict__ u, int B, double beta,
                                                         const uint8_t* __restrict__ done, const T* __restrict__ act,
                                                         const T* __restrict__ rew, int N, int A,
                                                         int64_t* __restrict__ rows, int64_t* __restrict__ index,
                                                         int64_t* __restrict__ stamp_out, int64_t* __restrict__ slot_out,
                                                         int64_t* __restrict__ env_out, uint8_t* __restrict__ done_out,
                                                         T* __restrict__ w_out, T* __restrict__ act_out,
                                                         T* __restrict__ rew_out) {
    const int lane = threadIdx.x & 31;
    const long long b = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (b >= B) return;
    const long long root = t.off[t.depth];
    const double total = t.sum[root];
    double x = u[b] * total, c_leaf = 0.0;
    long long node = 0;
    bool ok = true;
    for (int k = t.depth; k >= 1; --k) {
        const double c = child_sum(t, k - 1, node * 32 + lane);
        double P = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const double y = __shfl_up_sync(kFull, P, o);
            if (lane >= o) P += y;
        }
        double before = __shfl_up_sync(kFull, P, 1);
        if (lane == 0) before = 0.0;
        const unsigned pos = __ballot_sync(kFull, c > 0.0), hit = __ballot_sync(kFull, c > 0.0 && x < P);
        if (pos == 0u) { ok = false; break; }                // empty tree (warp-uniform)
        const int kk = hit ? __ffs(hit) - 1 : 31 - __clz(pos);
        const double ck = __shfl_sync(kFull, c, kk), pk = __shfl_sync(kFull, before, kk);
        x = fmax(x - pk, 0.0);
        if (!(x < ck)) x = nextafter(ck, 0.0);
        node = node * 32 + kk;
        c_leaf = ck;
    }
    const long long NA = (long long)N * A;
    if (!ok) {                                                // only when every leaf is 0
        if (lane == 0) {
            rows[b] = rows[B + b] = index[b] = stamp_out[b] = slot_out[b] = env_out[b] = -1;
            done_out[b] = 0;
            w_out[b] = (T)NAN;
        }
        for (long long i = lane; i < NA; i += 32) act_out[b * NA + i] = (T)NAN;
        for (long long i = lane; i < N; i += 32) rew_out[b * N + i] = (T)NAN;
        return;
    }
    const long long leaf = node, slot = leaf / t.E, e = leaf - slot * t.E;
    if (lane == 0) {
        const long long p = t.prev[slot];
        const uint8_t d = done[leaf];
        rows[b] = p >= 0 ? p * t.E + e : -1;
        rows[B + b] = d ? leaf + t.M : leaf;
        index[b] = leaf;
        stamp_out[b] = t.stamp[slot];
        slot_out[b] = slot;
        env_out[b] = e;
        done_out[b] = d;
        w_out[b] = (T)pow(t.mn[root] / c_leaf, beta);
    }
    for (long long i = lane; i < NA; i += 32) act_out[b * NA + i] = act[leaf * NA + i];
    for (long long i = lane; i < N; i += 32) rew_out[b * N + i] = rew[leaf * N + i];
}

// Recompute levels 1 .. depth above the leaf ranges [lo0, hi0] and, when `two`, [lo1, hi1].
void ancestors(const Tree& t, long long lo0, long long hi0, bool two, long long lo1, long long hi1, cudaStream_t st) {
    for (int k = 1; k <= t.depth; ++k) {
        const long long a0 = lo0 >> (5 * k), b0 = hi0 >> (5 * k);
        const long long a1 = two ? lo1 >> (5 * k) : 0, n1 = two ? (hi1 >> (5 * k)) - a1 + 1 : 0;
        const long long warps = (b0 - a0 + 1) + n1;
        k_per_level<<<grid_for(warps * 32), kThreads, 0, st>>>(t, k, nullptr, 0, a0, b0 - a0 + 1, a1, n1, nullptr, 0);
    }
}

template <typename T>
int per_sample_impl(const fg_per* p, const double* u, int B, double beta, const uint8_t* done, const void* actions,
                    const void* reward, int N, int A, int64_t* rows, int64_t* index, int64_t* stamp_out,
                    int64_t* slot_out, int64_t* env_out, uint8_t* done_out, void* weights, void* actions_out,
                    void* reward_out, void* stream, const char* who) {
    NvtxRange nvtx_(who);
    Tree t;
    int rc = make_tree(p, &t, who);
    if (rc) return rc;
    if (B < 1) return fail(FG_ERR_ARG, "%s: B must be >= 1", who);
    if (N < 1 || N > FG_MAX_AGENTS) return fail(FG_ERR_ARG, "%s: N must be in [1, FG_MAX_AGENTS=256]", who);
    if (A < 1 || A > 64) return fail(FG_ERR_ARG, "%s: A must be in [1, 64]", who);
    if (!(beta >= 0.0) || !std::isfinite(beta)) return fail(FG_ERR_ARG, "%s: beta must be finite and >= 0", who);
    if (!u || !done || !actions || !reward)
        return fail(FG_ERR_ARG, "%s: u / done / actions / reward must be non-null", who);
    if (!rows || !index || !stamp_out || !slot_out || !env_out || !done_out || !weights || !actions_out || !reward_out)
        return fail(FG_ERR_ARG, "%s: outputs must be non-null", who);
    if (!aligned(u, 8) || !aligned(rows, 8) || !aligned(index, 8) || !aligned(stamp_out, 8) || !aligned(slot_out, 8) ||
        !aligned(env_out, 8))
        return fail(FG_ERR_ARG, "%s: u and the int64 outputs must be 8-byte aligned", who);
    if (!aligned(actions, sizeof(T)) || !aligned(reward, sizeof(T)) || !aligned(weights, sizeof(T)) ||
        !aligned(actions_out, sizeof(T)) || !aligned(reward_out, sizeof(T)))
        return fail(FG_ERR_ARG, "%s: actions / reward / weights must be aligned to the real type", who);
    cudaStream_t st = (cudaStream_t)stream;
    k_per_sample<T><<<grid_for((long long)B * 32), kThreads, 0, st>>>(
        t, u, B, beta, done, (const T*)actions, (const T*)reward, N, A, rows, index, stamp_out, slot_out, env_out,
        done_out, (T*)weights, (T*)actions_out, (T*)reward_out);
    return launch_status(who);
}

template <typename TD>
void per_update_launch(const Tree& t, const int64_t* index, const int64_t* stamp, const void* td, int B, double alpha,
                       double eps, cudaStream_t st) {
    k_per_claim<TD><<<grid_for(B), kThreads, 0, st>>>(t, index, stamp, (const TD*)td, B);
    k_per_write<TD><<<grid_for(B), kThreads, 0, st>>>(t, index, (const TD*)td, B, alpha, eps);
}

}  // namespace

extern "C" {

int fg_per_layout(long long slots, long long envs, long long* nodes, int* depth, long long* scratch_bytes) {
    if (!nodes || !depth || !scratch_bytes)
        return fail(FG_ERR_ARG, "%s: nodes / depth / scratch_bytes must be non-null", "fg_per_layout");
    int rc = check_sizes(slots, envs, "fg_per_layout");
    if (rc) return rc;
    layout(slots * envs, nullptr, nodes, depth);
    *scratch_bytes = slots * envs * (long long)sizeof(int);
    return FG_OK;
}

int fg_per_fill(const fg_per* p, long long slot, long long prev, long long stamp, int valid, long long drop_slot,
                void* stream) {
    const char* who = "fg_per_fill";
    NvtxRange nvtx_(who);
    Tree t;
    int rc = make_tree(p, &t, who);
    if (rc) return rc;
    if (slot < 0 || slot >= t.T) return fail(FG_ERR_ARG, "%s: slot out of range", who);
    if (prev < -1 || prev >= t.T || prev == slot) return fail(FG_ERR_ARG, "%s: prev must be -1 or another slot", who);
    if (drop_slot < -1 || drop_slot >= t.T || drop_slot == slot)
        return fail(FG_ERR_ARG, "%s: drop_slot must be -1 or another slot", who);
    if (valid != 0 && valid != 1) return fail(FG_ERR_ARG, "%s: valid must be 0 or 1", who);
    if (valid && prev < 0) return fail(FG_ERR_ARG, "%s: a valid transition needs prev >= 0", who);
    if (stamp < 0) return fail(FG_ERR_ARG, "%s: stamp must be >= 0", who);
    int dev = 0, sms = 0;                                    // grid-stride fill: 8 CTAs per SM cover any E
    cudaError_t err = cudaGetDevice(&dev);
    if (err == cudaSuccess) err = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (err != cudaSuccess) {
        snprintf(fgabi::g_err, sizeof(fgabi::g_err), "%s: %s", who, cudaGetErrorString(err));
        return FG_ERR_CUDA;
    }
    cudaStream_t st = (cudaStream_t)stream;
    k_per_fill<<<grid_for(t.E, 8ll * sms), kThreads, 0, st>>>(t, slot, prev, stamp, valid, drop_slot);
    const bool two = drop_slot >= 0;
    ancestors(t, slot * t.E, slot * t.E + t.E - 1, two, two ? drop_slot * t.E : 0, two ? drop_slot * t.E + t.E - 1 : 0,
              st);
    return launch_status(who);
}

int fg_per_update(const fg_per* p, const int64_t* index, const int64_t* stamp, const void* td, int td_f64, int B,
                  double alpha, double eps, void* stream) {
    const char* who = "fg_per_update";
    NvtxRange nvtx_(who);
    Tree t;
    int rc = make_tree(p, &t, who);
    if (rc) return rc;
    if (B < 1) return fail(FG_ERR_ARG, "%s: B must be >= 1", who);
    if (!index || !stamp || !td) return fail(FG_ERR_ARG, "%s: index / stamp / td must be non-null", who);
    if (td_f64 != 0 && td_f64 != 1) return fail(FG_ERR_ARG, "%s: td_f64 must be 0 or 1", who);
    if (!aligned(index, 8) || !aligned(stamp, 8) || !aligned(td, td_f64 ? 8 : 4))
        return fail(FG_ERR_ARG, "%s: index / stamp / td must be aligned to their type", who);
    if (!(alpha >= 0.0) || !std::isfinite(alpha)) return fail(FG_ERR_ARG, "%s: alpha must be finite and >= 0", who);
    if (!(eps > 0.0) || !std::isfinite(eps)) return fail(FG_ERR_ARG, "%s: eps must be finite and > 0", who);
    cudaStream_t st = (cudaStream_t)stream;
    if (td_f64) per_update_launch<double>(t, index, stamp, td, B, alpha, eps, st);
    else per_update_launch<float>(t, index, stamp, td, B, alpha, eps, st);
    // a level with at most B nodes is recomputed whole (no node written twice); below that, one warp per entry
    for (int k = 1; k <= t.depth; ++k) {
        const bool whole = t.cnt[k] <= B;
        const long long warps = k == 1 ? B : (whole ? t.cnt[k] : B);      // (level 1 also resets the owners)
        k_per_level<<<grid_for(warps * 32), kThreads, 0, st>>>(t, k, whole ? nullptr : index, whole ? 0 : B, 0,
                                                           whole ? t.cnt[k] : 0, 0, 0, k == 1 ? index : nullptr,
                                                           k == 1 ? B : 0);
    }
    return launch_status(who);
}

int fg_per_sample(const fg_per* p, const double* u, int B, double beta, const uint8_t* done, const void* actions,
                  const void* reward, int N, int A, int64_t* rows, int64_t* index, int64_t* stamp_out,
                  int64_t* slot_out, int64_t* env_out, uint8_t* done_out, void* weights, void* actions_out,
                  void* reward_out, void* stream) {
    return per_sample_impl<float>(p, u, B, beta, done, actions, reward, N, A, rows, index, stamp_out, slot_out,
                                  env_out, done_out, weights, actions_out, reward_out, stream, "fg_per_sample");
}

int fg_per_sample_f64(const fg_per* p, const double* u, int B, double beta, const uint8_t* done, const void* actions,
                      const void* reward, int N, int A, int64_t* rows, int64_t* index, int64_t* stamp_out,
                      int64_t* slot_out, int64_t* env_out, uint8_t* done_out, void* weights, void* actions_out,
                      void* reward_out, void* stream) {
    return per_sample_impl<double>(p, u, B, beta, done, actions, reward, N, A, rows, index, stamp_out, slot_out,
                                   env_out, done_out, weights, actions_out, reward_out, stream, "fg_per_sample_f64");
}

}  // extern "C"
