// Graph construction kernels: segmented radius search, kNN graph, degree counts.
// Semantics of pytorch-cluster 1.6.1's CUDA kernels (see include/ddp_b200.h), redesigned as
// warp-per-query ordered scans (radius) and shared-memory-staged per-thread scans (kNN) that keep
// the exact fp32 arithmetic and the first-K-by-index / tie-by-index rules, with device-side edge
// counts (no host synchronisation) and a scan + compaction into fixed-capacity edge buffers.
#include "ddp_common.cuh"

namespace {

constexpr int kWarpsPerBlock = 8;

__global__ void radius_scan_kernel(const float *__restrict__ x, const float *__restrict__ y,
                                   const int32_t *__restrict__ ptr_x, const int32_t *__restrict__ ptr_y,
                                   int num_examples, int n_y, const float *__restrict__ inv_scale, float r2,
                                   int max_nbr, int graph_mode, int32_t *__restrict__ slab, int slab_w,
                                   int32_t *__restrict__ counts) {
    const int lane = threadIdx.x & 31;
    const int j = blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
    if (j >= n_y) return;
    const int b = ddp_find_segment(ptr_y, num_examples, j);
    float yx = y[3 * j], yy = y[3 * j + 1], yz = y[3 * j + 2];
    float c = 1.f;
    if (inv_scale != nullptr) {
        c = inv_scale[b];
        yx = __fdiv_rn(yx, c); yy = __fdiv_rn(yy, c); yz = __fdiv_rn(yz, c);
    }
    const int beg = ptr_x[b], end = ptr_x[b + 1];
    int cnt_all = 0, cnt_emit = 0;
    const unsigned lt = (1u << lane) - 1u;
    for (int base = beg; base < end && cnt_all < max_nbr; base += 32) {
        const int i = base + lane;
        bool hit = false;
        if (i < end) {
            float xx = x[3 * i], xy = x[3 * i + 1], xz = x[3 * i + 2];
            if (inv_scale != nullptr) { xx = __fdiv_rn(xx, c); xy = __fdiv_rn(xy, c); xz = __fdiv_rn(xz, c); }
            hit = ddp_sqdist(xx, xy, xz, yx, yy, yz) < r2;
        }
        const unsigned m_all = __ballot_sync(0xffffffffu, hit);
        const bool in_cap = hit && (cnt_all + __popc(m_all & lt) < max_nbr);
        const bool emit = in_cap && !(graph_mode && i == j);
        const unsigned m_emit = __ballot_sync(0xffffffffu, emit);
        if (emit) slab[(size_t)j * slab_w + cnt_emit + __popc(m_emit & lt)] = i;
        cnt_all += __popc(m_all);
        cnt_emit += __popc(m_emit);
    }
    if (lane == 0) counts[j] = cnt_emit;
}

template <int KP>
__device__ __forceinline__ void knn_insert(float (&bd)[KP], int (&bi)[KP], float d, int i) {
    if (bd[KP - 1] > d) {
        bd[KP - 1] = d; bi[KP - 1] = i;
#pragma unroll
        for (int e = KP - 1; e > 0; --e) {
            if (bd[e - 1] > bd[e]) {
                float td = bd[e - 1]; bd[e - 1] = bd[e]; bd[e] = td;
                int ti = bi[e - 1]; bi[e - 1] = bi[e]; bi[e] = ti;
            }
        }
    }
}

// Same list, candidates in arbitrary order: lexicographic (distance, index) comparison reproduces the scan's
// "ties keep the lower index" rule when partial lists are merged.
template <int KP>
__device__ __forceinline__ void knn_insert_lex(float (&bd)[KP], int (&bi)[KP], float d, int i) {
    if (bd[KP - 1] > d || (bd[KP - 1] == d && bi[KP - 1] > i)) {
        bd[KP - 1] = d; bi[KP - 1] = i;
#pragma unroll
        for (int e = KP - 1; e > 0; --e) {
            if (bd[e - 1] > bd[e] || (bd[e - 1] == bd[e] && bi[e - 1] > bi[e])) {
                float td = bd[e - 1]; bd[e - 1] = bd[e]; bd[e] = td;
                int ti = bi[e - 1]; bi[e - 1] = bi[e]; bi[e] = ti;
            }
        }
    }
}

constexpr int kKnnThreads = 128;
constexpr int kKnnSub = 4;       // threads per centre (each scans a quarter of the staged points, lists merged by shuffles)
constexpr int kKnnStage = 2048;  // points staged per pass (24 KB)

// kKnnSub threads per centre; the centre's example is staged through shared memory in chunks when the
// whole block lies inside one example (the common case), otherwise threads read global memory.
template <int KP>
__global__ void knn_scan_kernel(const float *__restrict__ x, const int32_t *__restrict__ ptr, int num_examples, int n,
                                int32_t *__restrict__ slab, int slab_w, int32_t *__restrict__ counts) {
    __shared__ float sx[kKnnStage * 3];
    constexpr int QPB = kKnnThreads / kKnnSub;      // centres per block
    const int sub = threadIdx.x % kKnnSub;
    const int j = blockIdx.x * QPB + threadIdx.x / kKnnSub;
    const int j_first = blockIdx.x * QPB;
    const int j_last = min(j_first + QPB, n) - 1;
    const int b_first = ddp_find_segment(ptr, num_examples, j_first);
    const int b_last = ddp_find_segment(ptr, num_examples, j_last);
    float bd[KP];
    int bi[KP];
#pragma unroll
    for (int e = 0; e < KP; ++e) { bd[e] = 1e10f; bi[e] = -1; }
    float yx = 0.f, yy = 0.f, yz = 0.f;
    if (j < n) { yx = x[3 * j]; yy = x[3 * j + 1]; yz = x[3 * j + 2]; }
    if (b_first == b_last) {
        const int beg = ptr[b_first], end = ptr[b_first + 1];
        for (int base = beg; base < end; base += kKnnStage) {
            const int m = min(kKnnStage, end - base);
            __syncthreads();
            for (int t = threadIdx.x; t < 3 * m; t += kKnnThreads) sx[t] = x[3 * base + t];
            __syncthreads();
            if (j < n) {
                const int per = (m + kKnnSub - 1) / kKnnSub;
                const int t1 = min(m, (sub + 1) * per);
                for (int t = sub * per; t < t1; ++t)
                    knn_insert<KP>(bd, bi, ddp_sqdist(sx[3 * t], sx[3 * t + 1], sx[3 * t + 2], yx, yy, yz), base + t);
            }
        }
    } else if (j < n) {
        const int b = ddp_find_segment(ptr, num_examples, j);
        const int beg = ptr[b], m = ptr[b + 1] - beg;
        const int per = (m + kKnnSub - 1) / kKnnSub;
        const int t1 = min(m, (sub + 1) * per);
        for (int t = sub * per; t < t1; ++t) {
            const int i = beg + t;
            knn_insert<KP>(bd, bi, ddp_sqdist(x[3 * i], x[3 * i + 1], x[3 * i + 2], yx, yy, yz), i);
        }
    }
    // merge the partial lists into the group's first thread (all lanes take part in the shuffles)
    const int lane = threadIdx.x & 31, lead = lane - sub;
#pragma unroll
    for (int s2 = 1; s2 < kKnnSub; ++s2) {
#pragma unroll
        for (int e = 0; e < KP; ++e) {
            const float d = __shfl_sync(0xffffffffu, bd[e], lead + s2);
            const int i = __shfl_sync(0xffffffffu, bi[e], lead + s2);
            if (sub == 0 && i != -1) knn_insert_lex<KP>(bd, bi, d, i);
        }
    }
    if (j < n && sub == 0) {
        int c = 0;
#pragma unroll
        for (int e = 0; e < KP; ++e) {
            if (bi[e] != -1 && bi[e] != j) { slab[(size_t)j * slab_w + c] = bi[e]; ++c; }
        }
        counts[j] = c;
    }
}

// Filtered form for small k on dense point sets (heavy atoms of a protein pocket) whose examples fit one shared-memory
// stage: kKnnFSub threads per centre scan a quarter of the example each and only RECORD the candidates closer than a
// radius (a rare, cheap event - no divergent sorted insertion inside the scan); the k + 1 nearest are then selected
// among the ~30 recorded ones with the (distance, index) order of the sequential scan.  Exact: if at least k + 1
// candidates lie inside the radius, the k + 1 nearest do too.  A centre with too few (surface atom) or too many
// recorded candidates retries with the next radius; the last resort is the full insertion scan.
constexpr int kKnnFilterCap = 96;
constexpr int kKnnFC = 32;           // centres per block
constexpr int kKnnFSub = 8;          // threads per centre (the scan is a latency-bound LDS -> FADD chain: more, shorter chains)
template <int KP>
__global__ void __launch_bounds__(kKnnFC * kKnnFSub)
knn_scan_filter_kernel(const float *__restrict__ x, const int32_t *__restrict__ ptr, int num_examples, int n,
                       int32_t *__restrict__ slab, int slab_w, int32_t *__restrict__ counts) {
    extern __shared__ __align__(16) unsigned char knn_smem[];
    float *sx = reinterpret_cast<float *>(knn_smem);                              // [kKnnStage * 3]
    int *cand = reinterpret_cast<int *>(sx + kKnnStage * 3);                       // [kKnnFilterCap][kKnnFC]
    int *cnt = cand + kKnnFilterCap * kKnnFC;                                      // [kKnnFC]
    const int tid = threadIdx.x, sub = tid % kKnnFSub, c = tid / kKnnFSub;
    // block -> (example, block inside the example): blocks never straddle examples (grid = ceil(n / FC) + num_examples)
    int b = 0, lb = blockIdx.x;
    while (b < num_examples) {
        const int nb = (ptr[b + 1] - ptr[b] + kKnnFC - 1) / kKnnFC;
        if (lb < nb) break;
        lb -= nb;
        ++b;
    }
    if (b >= num_examples) return;
    const int beg = ptr[b], m = ptr[b + 1] - beg;
    const int j0 = beg + lb * kKnnFC + c;
    const int j = j0 < beg + m ? j0 : n;                                           // n marks an idle lane
    float yx = 0.f, yy = 0.f, yz = 0.f;
    if (j < n) { yx = x[3 * j]; yy = x[3 * j + 1]; yz = x[3 * j + 2]; }
    if (m > kKnnStage) {                                                           // example too large to stage: plain scan
        if (j < n && sub == 0) {
            float bd[KP];
            int bi[KP];
#pragma unroll
            for (int e = 0; e < KP; ++e) { bd[e] = 1e10f; bi[e] = -1; }
            for (int i = beg; i < beg + m; ++i) knn_insert<KP>(bd, bi, ddp_sqdist(x[3 * i], x[3 * i + 1], x[3 * i + 2], yx, yy, yz), i);
            int o = 0;
#pragma unroll
            for (int e = 0; e < KP; ++e)
                if (bi[e] != -1 && bi[e] != j) { slab[(size_t)j * slab_w + o] = bi[e]; ++o; }
            counts[j] = o;
        }
        return;
    }
    for (int t = tid; t < 3 * m; t += kKnnFC * kKnnFSub) sx[t] = x[3 * beg + t];
    const int per = (m + kKnnFSub - 1) / kKnnFSub;
    const int q0 = sub * per, q1 = min(m, (sub + 1) * per);
    const unsigned group = ((1u << kKnnFSub) - 1u) << ((tid & 31) - sub);                              // the kKnnFSub lanes of this centre
    bool need = j < n;
    const float radii2[3] = {5.5f * 5.5f, 7.25f * 7.25f, 10.f * 10.f};      // sparse (surface) atoms retry with a wider ball
#pragma unroll 1
    for (int pass = 0; pass < 3; ++pass) {
        if (sub == 0) cnt[c] = 0;
        if (pass == 0) __syncthreads(); else __syncwarp(group);
        if (need) {
            const float r2 = radii2[pass];
            for (int t = q0; t < q1; ++t) {
                if (ddp_sqdist(sx[3 * t], sx[3 * t + 1], sx[3 * t + 2], yx, yy, yz) < r2) {
                    const int pos = atomicAdd(&cnt[c], 1);
                    if (pos < kKnnFilterCap) cand[pos * kKnnFC + c] = beg + t;
                }
            }
        }
        __syncwarp(group);
        const int got = cnt[c];
        // enough candidates (or simply every point of a tiny example) and no overflow: done
        need = need && !((got >= KP || got == m) && got <= kKnnFilterCap);
        if (!__any_sync(group, need)) break;
    }
    if (j >= n || sub != 0) return;
    float bd[KP];
    int bi[KP];
#pragma unroll
    for (int e = 0; e < KP; ++e) { bd[e] = 1e10f; bi[e] = -1; }
    if (!need) {
        const int got = cnt[c];
        for (int k = 0; k < got; ++k) {
            const int i = cand[k * kKnnFC + c] - beg;
            knn_insert_lex<KP>(bd, bi, ddp_sqdist(sx[3 * i], sx[3 * i + 1], sx[3 * i + 2], yx, yy, yz), beg + i);
        }
    } else {
        for (int t = 0; t < m; ++t) knn_insert<KP>(bd, bi, ddp_sqdist(sx[3 * t], sx[3 * t + 1], sx[3 * t + 2], yx, yy, yz), beg + t);
    }
    int o = 0;
#pragma unroll
    for (int e = 0; e < KP; ++e) {
        if (bi[e] != -1 && bi[e] != j) { slab[(size_t)j * slab_w + o] = bi[e]; ++o; }
    }
    counts[j] = o;
}

// Generic-k fallback (k + 1 <= 101, arrays in local memory).
__global__ void knn_scan_generic_kernel(const float *__restrict__ x, const int32_t *__restrict__ ptr, int num_examples,
                                        int n, int kp, int32_t *__restrict__ slab, int slab_w,
                                        int32_t *__restrict__ counts) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    float bd[101];
    int bi[101];
    for (int e = 0; e < kp; ++e) { bd[e] = 1e10f; bi[e] = -1; }
    const float yx = x[3 * j], yy = x[3 * j + 1], yz = x[3 * j + 2];
    const int b = ddp_find_segment(ptr, num_examples, j);
    for (int i = ptr[b]; i < ptr[b + 1]; ++i) {
        const float d = ddp_sqdist(x[3 * i], x[3 * i + 1], x[3 * i + 2], yx, yy, yz);
        for (int e1 = 0; e1 < kp; ++e1) {
            if (bd[e1] > d) {
                for (int e2 = kp - 1; e2 > e1; --e2) { bd[e2] = bd[e2 - 1]; bi[e2] = bi[e2 - 1]; }
                bd[e1] = d; bi[e1] = i;
                break;
            }
        }
    }
    int c = 0;
    for (int e = 0; e < kp; ++e)
        if (bi[e] != -1 && bi[e] != j) { slab[(size_t)j * slab_w + c] = bi[e]; ++c; }
    counts[j] = c;
}

// Exclusive scan of counts[0..n) in place (single block), counts[n] = total, *n_edges = prefix + total.
__global__ void scan_counts_kernel(int32_t *__restrict__ counts, int n, int prefix, int32_t *__restrict__ n_edges) {
    __shared__ int warp_sums[32];
    __shared__ int carry_s;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int base = 0; base < n; base += blockDim.x) {
        const int i = base + threadIdx.x;
        const int v = (i < n) ? counts[i] : 0;
        int s = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int t = __shfl_up_sync(0xffffffffu, s, o);
            if (lane >= o) s += t;
        }
        if (lane == 31) warp_sums[wid] = s;
        __syncthreads();
        if (wid == 0) {
            int w = (lane < (int)(blockDim.x >> 5)) ? warp_sums[lane] : 0;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                int t = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= o) w += t;
            }
            warp_sums[lane] = w;  // inclusive
        }
        __syncthreads();
        const int carry = carry_s;
        const int excl = carry + (wid > 0 ? warp_sums[wid - 1] : 0) + s - v;
        if (i < n) counts[i] = excl;
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) carry_s = carry + warp_sums[(blockDim.x >> 5) - 1];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        counts[n] = carry_s;
        *n_edges = prefix + carry_s;
    }
}

// C-alpha contact graph of datasets/process_mols.py:661-677, one warp per residue j of its complex: neighbours are
// the residues closer than r (index order); more than max_nbr of them -> the max_nbr nearest in ascending (distance,
// index) order instead; none -> the single nearest residue.  Fills slab[j][:counts[j]].  Distances in double from the
// fp32 coordinates, like the reference's scipy cdist, so that near-ties (ideal 3.8 A neighbours) order the same way.
__device__ __forceinline__ double calpha_dist(const float *__restrict__ pos, int i, double px, double py, double pz) {
    const double dx = (double)pos[3 * i] - px, dy = (double)pos[3 * i + 1] - py, dz = (double)pos[3 * i + 2] - pz;
    return __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz)));
}
__global__ void calpha_scan_kernel(const float *__restrict__ pos, const int32_t *__restrict__ ptr, int num_examples, int n,
                                   double r, int max_nbr, int32_t *__restrict__ slab, int slab_w, int32_t *__restrict__ counts) {
    const int lane = threadIdx.x & 31;
    const int j = blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
    if (j >= n) return;
    const int b = ddp_find_segment(ptr, num_examples, j);
    const int beg = ptr[b], end = ptr[b + 1];
    const double px = pos[3 * j], py = pos[3 * j + 1], pz = pos[3 * j + 2];
    const unsigned lt = (1u << lane) - 1u;
    int cnt = 0;
    for (int base = beg; base < end; base += 32) {
        const int i = base + lane;
        const bool hit = i < end && i != j && calpha_dist(pos, i, px, py, pz) < r;
        const unsigned m = __ballot_sync(0xffffffffu, hit);
        const int at = cnt + __popc(m & lt);
        if (hit && at < max_nbr) slab[(size_t)j * slab_w + at] = i;
        cnt += __popc(m);
    }
    int keep = cnt;
    if (cnt > max_nbr || cnt == 0) {
        keep = cnt == 0 ? 1 : max_nbr;
        if (keep > end - beg - 1) keep = end - beg - 1;
        double last_d = -1.0;
        int last_i = -1;
        for (int k = 0; k < keep; ++k) {
            double bd = INFINITY;
            int bi = 0x7fffffff;
            for (int i = beg + lane; i < end; i += 32) {
                if (i == j) continue;
                const double d = calpha_dist(pos, i, px, py, pz);
                const bool after = d > last_d || (d == last_d && i > last_i);
                if (after && (d < bd || (d == bd && i < bi))) { bd = d; bi = i; }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const double od = __shfl_xor_sync(0xffffffffu, bd, o);
                const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
                if (od < bd || (od == bd && oi < bi)) { bd = od; bi = oi; }
            }
            if (lane == 0) slab[(size_t)j * slab_w + k] = bi;
            last_d = bd; last_i = bi;
        }
    }
    if (lane == 0) counts[j] = keep;
}

__global__ void compact_edges_kernel(const int32_t *__restrict__ slab, int slab_w, const int32_t *__restrict__ offs,
                                     int n_y, int swap_rows, int prefix, int32_t *__restrict__ edge, int edge_cap) {
    const int lane = threadIdx.x & 31;
    const int j = blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
    if (j >= n_y) return;
    const int o = offs[j], c = offs[j + 1] - o;
    for (int t = lane; t < c; t += 32) {
        const int e = prefix + o + t;
        if (e < edge_cap) {
            const int i = slab[(size_t)j * slab_w + t];
            edge[e] = swap_rows ? i : j;
            edge[edge_cap + e] = swap_rows ? j : i;
        }
    }
}

__global__ void degree_kernel(const int32_t *__restrict__ idx, const int32_t *__restrict__ n_edges, int32_t *__restrict__ deg) {
    const int n = *n_edges;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) atomicAdd(&deg[idx[e]], 1);
}

// live[i] = 1 if node i is an endpoint of one of its example's bonds or (r2 > 0) lies closer than sqrt(r2) to the midpoint
// of one, else 0 (every entry is written).  The midpoint is formed as in bond_geometry_kernel (embed.cu).
__global__ void mark_bond_nodes_kernel(const float *__restrict__ pos, const int32_t *__restrict__ node_ptr, int num_examples, int n,
                                       const int32_t *__restrict__ bonds, int n_bonds, const int32_t *__restrict__ bond_ptr,
                                       float r2, uint8_t *__restrict__ live) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint8_t hit = 0;
    if (n_bonds > 0) {
        const int b = ddp_find_segment(node_ptr, num_examples, i);
        const float px = pos[3 * i], py = pos[3 * i + 1], pz = pos[3 * i + 2];
        for (int k = bond_ptr[b]; k < bond_ptr[b + 1] && !hit; ++k) {
            const int u = bonds[k], v = bonds[n_bonds + k];
            hit = u == i || v == i;
            if (!hit && r2 > 0.f)
                hit = ddp_sqdist(px, py, pz, (pos[3 * u] + pos[3 * v]) / 2.f, (pos[3 * u + 1] + pos[3 * v + 1]) / 2.f,
                                 (pos[3 * u + 2] + pos[3 * v + 2]) / 2.f) < r2;
        }
    }
    live[i] = hit;
}

// live_out[gather[e]] = 1 for every live edge e whose aggregation node is live in live_in (every edge: live_in == NULL)
__global__ void mark_gathered_kernel(const int32_t *__restrict__ agg, const int32_t *__restrict__ gather,
                                     const int32_t *__restrict__ n_edges, int edge_cap, const uint8_t *__restrict__ live_in,
                                     uint8_t *__restrict__ live_out) {
    const int n = min(*n_edges, edge_cap);
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x)
        if (live_in == nullptr || live_in[agg[e]]) live_out[gather[e]] = 1;
}

// Stable compaction of the edges whose aggregation node is live: count per block of kCompactBlock edges, exclusive scan of
// the counts (scan_counts_kernel), then every block writes its live edges in order from its offset.
constexpr int kCompactBlock = 256;
__device__ __forceinline__ bool edge_is_live(const int32_t *__restrict__ agg, const int32_t *__restrict__ n_edges, int edge_cap,
                                             const uint8_t *__restrict__ live, int e) {
    return e < min(*n_edges, edge_cap) && live[agg[e]];
}

__global__ void __launch_bounds__(kCompactBlock) live_count_kernel(const int32_t *__restrict__ agg, const int32_t *__restrict__ n_edges,
                                                                   int edge_cap, const uint8_t *__restrict__ live, int32_t *__restrict__ counts) {
    const int c = __syncthreads_count(edge_is_live(agg, n_edges, edge_cap, live, blockIdx.x * kCompactBlock + threadIdx.x));
    if (threadIdx.x == 0) counts[blockIdx.x] = c;
}

__global__ void __launch_bounds__(kCompactBlock) live_scatter_kernel(
        const int32_t *__restrict__ edge, int edge_cap, const int32_t *__restrict__ n_edges, int agg_row,
        const float *__restrict__ sh, int sh_dim, const float *__restrict__ emb, int ns, const uint8_t *__restrict__ live,
        const int32_t *__restrict__ offs, int32_t *__restrict__ edge_out, int edge_cap_out, float *__restrict__ sh_out,
        float *__restrict__ emb_out) {
    __shared__ int warp_off[kCompactBlock / 32];
    __shared__ int src[kCompactBlock];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int e = blockIdx.x * kCompactBlock + threadIdx.x;
    const bool keep = edge_is_live(edge + (size_t)agg_row * edge_cap, n_edges, edge_cap, live, e);
    const unsigned m = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) warp_off[wid] = __popc(m);
    __syncthreads();
    int before = 0, total = 0;
#pragma unroll
    for (int w = 0; w < kCompactBlock / 32; ++w) {
        before += w < wid ? warp_off[w] : 0;
        total += warp_off[w];
    }
    const int local = before + __popc(m & ((1u << lane) - 1u));
    const int base = offs[blockIdx.x];
    if (keep) {
        src[local] = e;
        edge_out[base + local] = edge[e];
        edge_out[edge_cap_out + base + local] = edge[edge_cap + e];
    }
    __syncthreads();
    // rows of the kept edges, copied by the whole block (consecutive threads -> consecutive floats)
    for (int t = threadIdx.x; t < total * sh_dim; t += kCompactBlock) {
        const int k = t / sh_dim, c = t - k * sh_dim;
        sh_out[(size_t)(base + k) * sh_dim + c] = sh[(size_t)src[k] * sh_dim + c];
    }
    for (int t = threadIdx.x; t < total * ns; t += kCompactBlock) {
        const int k = t / ns, c = t - k * ns;
        emb_out[(size_t)(base + k) * ns + c] = emb[(size_t)src[k] * ns + c];
    }
}

constexpr int kMaxDegJobs = 12;
struct DegPack { ddp_degree_job_t j[kMaxDegJobs]; };
__global__ void degree_multi_kernel(DegPack p) {
    const ddp_degree_job_t j = p.j[blockIdx.y];
    const int n = min(*j.n_edges_dev, j.edge_cap);
    for (int e = j.start + blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) atomicAdd(&j.deg[j.idx[e]], 1);
}

}  // namespace

extern "C" int ddp_radius(const float *x, const float *y, const int32_t *ptr_x, const int32_t *ptr_y,
                          int32_t num_examples, int32_t n_y, const float *inv_scale, float r, int32_t max_nbr,
                          int32_t mode, int32_t prefix, int32_t *slab, int32_t slab_w, int32_t *counts,
                          int32_t *edge, int32_t edge_cap, int32_t *n_edges_dev, void *stream) {
    if (!x || !y || !ptr_x || !ptr_y || !slab || !counts || !edge || !n_edges_dev) return DDP_E_ARG;
    if (num_examples <= 0 || n_y < 0 || max_nbr <= 0 || slab_w <= 0 || prefix < 0) return DDP_E_SHAPE;
    cudaStream_t st = (cudaStream_t)stream;
    const float r2 = (float)((double)r * (double)r);
    if (n_y > 0) {
        radius_scan_kernel<<<(n_y + kWarpsPerBlock - 1) / kWarpsPerBlock, kWarpsPerBlock * 32, 0, st>>>(
            x, y, ptr_x, ptr_y, num_examples, n_y, inv_scale, r2, max_nbr, mode & DDP_RADIUS_GRAPH, slab, slab_w, counts);
        DDP_LAUNCH_CHECK();
    }
    scan_counts_kernel<<<1, 1024, 0, st>>>(counts, n_y, prefix, n_edges_dev);
    DDP_LAUNCH_CHECK();
    if (n_y > 0) {
        compact_edges_kernel<<<(n_y + kWarpsPerBlock - 1) / kWarpsPerBlock, kWarpsPerBlock * 32, 0, st>>>(
            slab, slab_w, counts, n_y, mode & DDP_RADIUS_GRAPH, prefix, edge, edge_cap);
        DDP_LAUNCH_CHECK();
    }
    return 0;
}

extern "C" int ddp_knn_graph(const float *x, const int32_t *ptr, int32_t num_examples, int32_t n, int32_t k,
                             int32_t *slab, int32_t slab_w, int32_t *counts, int32_t *edge, int32_t edge_cap,
                             int32_t *n_edges_dev, void *stream) {
    if (!x || !ptr || !slab || !counts || !edge || !n_edges_dev) return DDP_E_ARG;
    if (num_examples <= 0 || n < 0 || k <= 0 || k > 100 || slab_w < k + 1) return DDP_E_SHAPE;
    cudaStream_t st = (cudaStream_t)stream;
    const int kp = k + 1;
    if (n > 0) {
        const int qpb = kKnnThreads / kKnnSub;
        const int grid_sub = (n + qpb - 1) / qpb, grid = (n + kKnnThreads - 1) / kKnnThreads;
        const size_t fsm = (size_t)kKnnStage * 3 * sizeof(float) + (size_t)(kKnnFilterCap + 1) * kKnnFC * sizeof(int);
        static bool configured9[DDP_MAX_DEVICES] = {false}, configured13[DDP_MAX_DEVICES] = {false};
        cudaError_t e1 = ddp_smem_opt_in(knn_scan_filter_kernel<9>, fsm, configured9);
        cudaError_t e2 = ddp_smem_opt_in(knn_scan_filter_kernel<13>, fsm, configured13);
        if (e1 != cudaSuccess || e2 != cudaSuccess) return (int)(e1 != cudaSuccess ? e1 : e2);
        const bool filt = kp == 9 || kp == 13;
        const int fgrid = (n + kKnnFC - 1) / kKnnFC + num_examples;
        if (filt && kp == 9) knn_scan_filter_kernel<9><<<fgrid, kKnnFC * kKnnFSub, fsm, st>>>(x, ptr, num_examples, n, slab, slab_w, counts);
        else if (filt) knn_scan_filter_kernel<13><<<fgrid, kKnnFC * kKnnFSub, fsm, st>>>(x, ptr, num_examples, n, slab, slab_w, counts);
        else if (kp == 9) knn_scan_kernel<9><<<grid_sub, kKnnThreads, 0, st>>>(x, ptr, num_examples, n, slab, slab_w, counts);
        else if (kp == 13) knn_scan_kernel<13><<<grid_sub, kKnnThreads, 0, st>>>(x, ptr, num_examples, n, slab, slab_w, counts);
        else if (kp == 33) knn_scan_kernel<33><<<grid_sub, kKnnThreads, 0, st>>>(x, ptr, num_examples, n, slab, slab_w, counts);
        else knn_scan_generic_kernel<<<grid, kKnnThreads, 0, st>>>(x, ptr, num_examples, n, kp, slab, slab_w, counts);
        DDP_LAUNCH_CHECK();
    }
    scan_counts_kernel<<<1, 1024, 0, st>>>(counts, n, 0, n_edges_dev);
    DDP_LAUNCH_CHECK();
    if (n > 0) {
        compact_edges_kernel<<<(n + kWarpsPerBlock - 1) / kWarpsPerBlock, kWarpsPerBlock * 32, 0, st>>>(
            slab, slab_w, counts, n, 1, 0, edge, edge_cap);
        DDP_LAUNCH_CHECK();
    }
    return 0;
}

extern "C" int ddp_calpha_graph(const float *pos, const int32_t *ptr, int32_t num_examples, int32_t n, float r, int32_t max_nbr,
                                int32_t *slab, int32_t slab_w, int32_t *counts, int32_t *edge, int32_t edge_cap,
                                int32_t *n_edges_dev, void *stream) {
    if (!pos || !ptr || !slab || !counts || !edge || !n_edges_dev) return DDP_E_ARG;
    if (num_examples <= 0 || n < 0 || max_nbr <= 0 || slab_w < max_nbr) return DDP_E_SHAPE;
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = (n + kWarpsPerBlock - 1) / kWarpsPerBlock;
    if (n > 0) {
        calpha_scan_kernel<<<grid, kWarpsPerBlock * 32, 0, st>>>(pos, ptr, num_examples, n, (double)r, max_nbr, slab, slab_w, counts);
        DDP_LAUNCH_CHECK();
    }
    scan_counts_kernel<<<1, 1024, 0, st>>>(counts, n, 0, n_edges_dev);
    DDP_LAUNCH_CHECK();
    if (n > 0) {
        compact_edges_kernel<<<grid, kWarpsPerBlock * 32, 0, st>>>(slab, slab_w, counts, n, 0, 0, edge, edge_cap);
        DDP_LAUNCH_CHECK();
    }
    return 0;
}

extern "C" int ddp_degree(const int32_t *idx, const int32_t *n_edges_dev, int32_t edge_cap, int32_t *deg, void *stream) {
    if (!idx || !n_edges_dev || !deg) return DDP_E_ARG;
    if (edge_cap <= 0) return 0;
    int grid = (edge_cap + 255) / 256;
    if (grid > 4 * ddp_num_sms()) grid = 4 * ddp_num_sms();
    degree_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(idx, n_edges_dev, deg);
    DDP_LAUNCH_CHECK();
    return 0;
}

extern "C" int ddp_degree_multi(const ddp_degree_job_t *jobs_host, int32_t n_jobs, void *stream) {
    if (!jobs_host || n_jobs < 0 || n_jobs > kMaxDegJobs) return DDP_E_ARG;
    if (n_jobs == 0) return 0;
    DegPack p;
    int cap = 0;
    for (int i = 0; i < n_jobs; ++i) {
        if (!jobs_host[i].idx || !jobs_host[i].n_edges_dev || !jobs_host[i].deg || jobs_host[i].start < 0) return DDP_E_ARG;
        p.j[i] = jobs_host[i];
        cap = jobs_host[i].edge_cap > cap ? jobs_host[i].edge_cap : cap;
    }
    if (cap <= 0) return 0;
    int gx = (cap + 255) / 256;
    if (gx > 2 * ddp_num_sms()) gx = 2 * ddp_num_sms();
    degree_multi_kernel<<<dim3(gx, n_jobs), 256, 0, (cudaStream_t)stream>>>(p);
    DDP_LAUNCH_CHECK();
    return 0;
}

extern "C" int ddp_mark_bond_nodes(const float *pos, const int32_t *node_ptr, int32_t num_examples, int32_t n,
                                   const int32_t *bonds, int32_t n_bonds, const int32_t *bond_ptr, float r, uint8_t *live,
                                   void *stream) {
    if (!pos || !node_ptr || !live || (n_bonds > 0 && (!bonds || !bond_ptr))) return DDP_E_ARG;
    if (num_examples <= 0 || n < 0 || n_bonds < 0) return DDP_E_SHAPE;
    if (n == 0) return 0;
    const float r2 = r > 0.f ? (float)((double)r * (double)r) : 0.f;
    mark_bond_nodes_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(pos, node_ptr, num_examples, n, bonds, n_bonds,
                                                                              bond_ptr, r2, live);
    DDP_LAUNCH_CHECK();
    return 0;
}

extern "C" int ddp_mark_gathered(const int32_t *agg, const int32_t *gather, const int32_t *n_edges_dev, int32_t edge_cap,
                                 const uint8_t *live_in, uint8_t *live_out, void *stream) {
    if (!gather || !n_edges_dev || !live_out || (live_in && !agg)) return DDP_E_ARG;
    if (edge_cap <= 0) return 0;
    int grid = (edge_cap + 255) / 256;
    if (grid > 4 * ddp_num_sms()) grid = 4 * ddp_num_sms();
    mark_gathered_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(agg, gather, n_edges_dev, edge_cap, live_in, live_out);
    DDP_LAUNCH_CHECK();
    return 0;
}

extern "C" int ddp_live_edges(const int32_t *edge, int32_t edge_cap, const int32_t *n_edges_dev, int32_t agg_row,
                              const float *sh, int32_t sh_dim, const float *emb, int32_t ns, const uint8_t *live,
                              int32_t *counts, int32_t *edge_out, int32_t edge_cap_out, int32_t *n_edges_out_dev,
                              float *sh_out, float *emb_out, void *stream) {
    if (!edge || !n_edges_dev || !sh || !emb || !live || !counts || !edge_out || !n_edges_out_dev || !sh_out || !emb_out)
        return DDP_E_ARG;
    if (edge_cap <= 0 || edge_cap_out < edge_cap || (agg_row != 0 && agg_row != 1) || sh_dim <= 0 || ns <= 0) return DDP_E_SHAPE;
    cudaStream_t st = (cudaStream_t)stream;
    const int blocks = (edge_cap + kCompactBlock - 1) / kCompactBlock;
    const int32_t *agg = edge + (size_t)agg_row * edge_cap;
    live_count_kernel<<<blocks, kCompactBlock, 0, st>>>(agg, n_edges_dev, edge_cap, live, counts);
    DDP_LAUNCH_CHECK();
    scan_counts_kernel<<<1, 1024, 0, st>>>(counts, blocks, 0, n_edges_out_dev);
    DDP_LAUNCH_CHECK();
    live_scatter_kernel<<<blocks, kCompactBlock, 0, st>>>(edge, edge_cap, n_edges_dev, agg_row, sh, sh_dim, emb, ns, live, counts,
                                                          edge_out, edge_cap_out, sh_out, emb_out);
    DDP_LAUNCH_CHECK();
    return 0;
}
