// Tracks from pairwise feature matches (sfm_build_tracks): the connected components of the match graph on the N
// features of V views, each component of two or more features one track.
//
// Semantics (include/sfm_b200.h):
//   features   view v owns the global ids [off[v], off[v+1]); local feature i of v is off[v] + i; N = off[V] <= INT32_MAX.
//   edges      every match (i, j) of a pair entry (a, b) is the undirected edge {off[a] + i, off[b] + j}; only the edge
//              set matters (order, multiplicity, direction and the grouping into pair entries do not).
//   tracks     components of >= 2 features, ordered by their smallest global id; observations in ascending global id
//              (by view, then by local index).  CONFLICT when two observations share a view (adjacent in that order),
//              else LONG when there are more than SFM_TRACK_MAX_OBSERVATIONS, else OK.
//
// Mapping (one call, every launch on the context's stream):
//   k_tb_init      parent[g] = g, size[g] = 0, track[g] = -1.
//   k_tb_hook      one thread per match: the roots of both ends, then atomicCAS(parent[hi], hi, lo) until they agree
//                  (the min-label hooking of ECL-CC, Jaiganesh and Burtscher, HPDC 2018).  Invariant parent[g] <= g: a
//                  root is its component's minimum, so the final labels do not depend on scheduling, and every find
//                  terminates.  Finds halve paths.  parent is read through relaxed device-scope atomics: a plain load
//                  may be served stale from L1, and a CAS retried against a stale root would never succeed.
//   k_tb_compress  a separate launch (hooking has finished): label[g] = root, size[root] += 1.  The root goes to its
//                  own array: a find racing through g may still store an older ancestor into parent[g].
//   k_tb_flag      flag[g] = (size of g's component >= 2).
//   cub scan       inclusive sum of flag: the slot of each selected feature, plus one; M = its last entry (read back:
//                  the sort needs it on the host).
//   k_tb_select    the selected features in id order with their labels: key[slot] = label, id[slot] = g.
//   cub sort       stable radix sort of (label, id) over the bits of N - 1: by label, then by id.
//   k_tb_heads     head[i] = the i-th sorted observation starts a track.
//   cub scan       inclusive sum of head: the track of each observation, plus one.
//   k_tb_obs       view (binary search of off), feature, the track scatter, offsets at heads, and a CONFLICT mark
//                  when an observation's view equals its predecessor's in the same track; the last one writes T and
//                  offsets[T] = M.
//   k_tb_status    per track: CONFLICT as marked, else LONG above SFM_TRACK_MAX_OBSERVATIONS, else OK.
#pragma once
#include <cuda/atomic>

#include <cstdint>

namespace sfm {

constexpr int kTbBlock = 256;
enum { TB_OK = 0, TB_CONFLICT = 1, TB_LONG = 2 };
constexpr int kTbMaxObservations = 64;  // SFM_TRACK_MAX_OBSERVATIONS

// One pair entry as the hook kernel reads it: the global ids of the first features of its two views.
struct TbPair {
    int base_a, base_b;
};

// ---- union-find, host and device (tools/track_build_check.cu runs these on CPU threads) -----------------------------
__host__ __device__ inline int tb_load(int* p) {
    return cuda::atomic_ref<int, cuda::thread_scope_device>(*p).load(cuda::std::memory_order_relaxed);
}

// The root of x.  Each visited node is pointed at its grandparent (path halving); that value is an ancestor of x in the
// same component and below it, so a racing store keeps parent[g] <= g and the component unchanged.
__host__ __device__ inline int tb_find(int* parent, int x) {
    int p = tb_load(parent + x);
    while (p != x) {
        const int g = tb_load(parent + p);
        if (g != p) cuda::atomic_ref<int, cuda::thread_scope_device>(parent[x]).store(g, cuda::std::memory_order_relaxed);
        x = p;
        p = g;
    }
    return x;
}

// Join the components of u and v: hook the larger root under the smaller until both finds agree.
__host__ __device__ inline void tb_hook(int* parent, int u, int v) {
    int ru = tb_find(parent, u), rv = tb_find(parent, v);
    while (ru != rv) {
        const int hi = ru > rv ? ru : rv, lo = ru > rv ? rv : ru;
        int expected = hi;
        if (cuda::atomic_ref<int, cuda::thread_scope_device>(parent[hi]).compare_exchange_strong(
                expected, lo, cuda::std::memory_order_relaxed))
            return;
        // hi was hooked by another thread meanwhile: start again from its new parent
        ru = tb_find(parent, expected);
        rv = tb_find(parent, lo);
    }
}

// The view owning global id g: the last v with off[v] <= g (views without features are skipped).
__host__ __device__ inline int tb_view_of(const long long* off, int V, long long g) {
    int lo = 0, hi = V;  // off[lo] <= g < off[hi]
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (off[mid] <= g) lo = mid;
        else hi = mid;
    }
    return lo;
}

#ifdef __CUDACC__
struct TbArgs {
    int N, V;
    long long E, P;
    const long long* foff;    // [V+1]
    const long long* moff;    // [P+1]
    const TbPair* pairs;      // [P]
    const int2* matches;      // [E]
    int* parent;              // [N]
    int* label;               // [N] the root of every feature, after k_tb_compress
    int* size;                // [N]
    int* flag;                // [N]
    int* track;               // [N]
};

__global__ void k_tb_init(TbArgs a) {
    for (long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x; g < a.N; g += (long long)gridDim.x * blockDim.x) {
        a.parent[g] = (int)g;
        a.size[g] = 0;
        a.track[g] = -1;
    }
}

__global__ void k_tb_hook(TbArgs a) {
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < a.E; e += (long long)gridDim.x * blockDim.x) {
        long long lo = 0, hi = a.P;  // the pair entry of match e: moff[lo] <= e < moff[hi]
        while (hi - lo > 1) {
            const long long mid = (lo + hi) >> 1;
            if (__ldg(a.moff + mid) <= e) lo = mid;
            else hi = mid;
        }
        const TbPair p = a.pairs[lo];
        const int2 m = __ldg(a.matches + e);
        tb_hook(a.parent, p.base_a + m.x, p.base_b + m.y);
    }
}

__global__ void k_tb_compress(TbArgs a) {
    for (long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x; g < a.N; g += (long long)gridDim.x * blockDim.x) {
        const int r = tb_find(a.parent, (int)g);
        a.label[g] = r;
        atomicAdd(a.size + r, 1);
    }
}

__global__ void k_tb_flag(TbArgs a) {
    for (long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x; g < a.N; g += (long long)gridDim.x * blockDim.x)
        a.flag[g] = a.size[a.label[g]] >= 2;
}

// pos: the inclusive sum of flag
__global__ void k_tb_select(TbArgs a, const int* __restrict__ pos, unsigned* __restrict__ key, unsigned* __restrict__ id) {
    for (long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x; g < a.N; g += (long long)gridDim.x * blockDim.x)
        if (a.flag[g]) {
            const int i = pos[g] - 1;
            key[i] = (unsigned)a.label[g];
            id[i] = (unsigned)g;
        }
}

__global__ void k_tb_heads(const unsigned* __restrict__ key, int M, int* __restrict__ head) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < M; i += (long long)gridDim.x * blockDim.x)
        head[i] = i == 0 || key[i] != key[i - 1];
}

// One thread per observation of the sorted order; tix[i] - 1 is its track.  status[] reads 0 on entry for every track.
__global__ void k_tb_obs(const long long* __restrict__ foff, int V, const unsigned* __restrict__ id, const int* __restrict__ tix,
                         int M, long long* __restrict__ offsets, int* __restrict__ status, int* __restrict__ view,
                         int* __restrict__ feature, int* __restrict__ track, int* __restrict__ T_out) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < M; i += (long long)gridDim.x * blockDim.x) {
        const int t = tix[i] - 1;
        const int g = (int)id[i];
        const int v = tb_view_of(foff, V, g);
        view[i] = v;
        feature[i] = g;
        track[g] = t;
        if (i == 0 || tix[i - 1] != tix[i]) offsets[t] = i;
        else if (tb_view_of(foff, V, (int)id[i - 1]) == v) status[t] = TB_CONFLICT;  // every writer writes the same
        if (i == M - 1) {
            offsets[t + 1] = M;
            *T_out = t + 1;
        }
    }
}

__global__ void k_tb_status(const long long* __restrict__ offsets, int T, int* __restrict__ status) {
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < T; t += (long long)gridDim.x * blockDim.x)
        if (status[t] != TB_CONFLICT) status[t] = offsets[t + 1] - offsets[t] > kTbMaxObservations ? TB_LONG : TB_OK;
}
#endif

}  // namespace sfm
