// Small (HBM / latency bound) kernels around the convolutions: sigma embedding + per-graph
// projections, node initialisation, fused edge geometry + spherical harmonics + radial basis +
// edge-embedding MLP, node update (scatter-mean + BatchNorm + residual), heads.
#include "ddp_common.cuh"

namespace {

// ---------------------------------------------------------------------------------------------
__global__ void graph_sigma_proj_kernel(const float *__restrict__ t, float scale, const float *__restrict__ freq,
                                        int sig_dim, const float *__restrict__ w, const float *__restrict__ b,
                                        int n_graphs, int ns, float *__restrict__ sig, float *__restrict__ out) {
    extern __shared__ float s_sig[];
    const int g = blockIdx.x, m = blockIdx.y;
    const int half = sig_dim / 2;
    for (int i = threadIdx.x; i < sig_dim; i += blockDim.x) {
        float v = 0.f;
        if (i < 2 * half) {
            const float arg = __fmul_rn(__fmul_rn(scale, t[g]), freq[i < half ? i : i - half]);
            v = (i < half) ? sinf(arg) : cosf(arg);
        }
        s_sig[i] = v;
        if (m == 0) sig[(size_t)g * sig_dim + i] = v;
    }
    __syncthreads();
    for (int o = threadIdx.x; o < ns; o += blockDim.x) {
        const float *wm = w + (size_t)m * sig_dim * ns;
        float acc = b[(size_t)m * ns + o];
        for (int k = 0; k < sig_dim; ++k) acc = fmaf(wm[(size_t)k * ns + o], s_sig[k], acc);
        out[((size_t)m * n_graphs + g) * ns + o] = acc;
    }
}

__global__ void node_init_kernel(const float *__restrict__ sp, const float *__restrict__ u,
                                 const int32_t *__restrict__ graph_of, int n, int ns, float *__restrict__ out, int ld) {
    const size_t total = (size_t)n * ns;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int node = (int)(i / ns), c = (int)(i % ns);
        out[(size_t)node * ld + c] = sp[i] + u[(size_t)graph_of[node] * ns + c];
    }
}

// ---------------------------------------------------------------------------------------------
// Static (time-independent) part of AtomEncoder (models/score_model.py:74-82), once per complex:
//   out[n][:] = (sum_k Emb_k[cat[n][k]]) W_emb + lm[n][:] W_lm
// One block per node: the summed embedding row and the language-model row (1280 floats) are staged in shared memory,
// thread o accumulates output channel o over K with weight reads coalesced across the block.
constexpr int kStaticThreads = 64;
__global__ void __launch_bounds__(kStaticThreads)
node_static_embed_kernel(const int64_t *__restrict__ cat, int n_cat, const float *__restrict__ table,
                         const int32_t *__restrict__ table_off, const float *__restrict__ lm, int n_lm,
                         const float *__restrict__ w_emb_t, const float *__restrict__ w_lm_t, int ns,
                         float *__restrict__ out) {
    extern __shared__ float s_row[];               // [ns | n_lm]
    const int node = blockIdx.x, tid = threadIdx.x;
    for (int c = tid; c < ns; c += kStaticThreads) {
        float h = 0.f;
        for (int k = 0; k < n_cat; ++k)            // same summation order as the reference loop over the embedding tables
            h += table[((size_t)table_off[k] + (size_t)cat[(size_t)node * n_cat + k]) * ns + c];
        s_row[c] = h;
    }
    for (int k = tid; k < n_lm; k += kStaticThreads) s_row[ns + k] = lm[(size_t)node * n_lm + k];
    __syncthreads();
    for (int o = tid; o < ns; o += kStaticThreads) {
        float a0 = 0.f, a1 = 0.f;
        if (w_emb_t != nullptr) {
            for (int k = 0; k < ns; ++k) a0 = fmaf(s_row[k], __ldg(w_emb_t + (size_t)k * ns + o), a0);
        } else {
            a0 = s_row[o];                         // no Linear over the embedding sum (OldAtomEncoder without LM features)
        }
        int k = 0;
        for (; k + 1 < n_lm; k += 2) {             // two chains: 1280 dependent FMAs would be latency bound
            a0 = fmaf(s_row[ns + k], __ldg(w_lm_t + (size_t)k * ns + o), a0);
            a1 = fmaf(s_row[ns + k + 1], __ldg(w_lm_t + (size_t)(k + 1) * ns + o), a1);
        }
        if (k < n_lm) a0 = fmaf(s_row[ns + k], __ldg(w_lm_t + (size_t)k * ns + o), a0);
        out[(size_t)node * ns + o] = a0 + a1;
    }
}

// ---------------------------------------------------------------------------------------------
// Edge geometry + embedding: 32 edges per block, 128 threads = 2 edge halves x 64 output lanes.
constexpr int kEE = 32;
constexpr int kEEThreads = 128;
constexpr int kMaxNs = 64, kMaxRbf = 64, kMaxPre = 8;

__global__ void __launch_bounds__(kEEThreads)
edge_embed_kernel(const float *__restrict__ pos_a, const float *__restrict__ pos_b, const int32_t *__restrict__ edge,
                  int cap, const int32_t *__restrict__ n_edges_dev, const int32_t *__restrict__ graph_of_a,
                  const float *__restrict__ pre, int n_pre_rows, const float *__restrict__ u, ddp_edge_mlp_t p,
                  float *__restrict__ sh_out, float *__restrict__ emb) {
    __shared__ float s_in[(kMaxRbf + kMaxPre) * kEE];   // [k][edge]
    __shared__ float s_r[kMaxNs * kEE];                 // [j][edge]
    __shared__ float s_d[kEE];
    __shared__ int s_g[kEE];
    const int n_edges = min(*n_edges_dev, cap);
    const int e0 = blockIdx.x * kEE;
    if (e0 >= n_edges) return;
    const int tid = threadIdx.x;
    if (tid < kEE) {
        const int e = e0 + tid;
        float d = 0.f;
        int g = 0;
        if (e < n_edges) {
            const int a = edge[e], b = edge[cap + e];
            const float vx = pos_b[3 * b] - pos_a[3 * a], vy = pos_b[3 * b + 1] - pos_a[3 * a + 1],
                        vz = pos_b[3 * b + 2] - pos_a[3 * a + 2];
            d = sqrtf(vx * vx + vy * vy + vz * vz);
            const float inv = 1.f / fmaxf(d, 1e-12f);
            const float x = vx * inv, y = vy * inv, z = vz * inv;
            const float s3 = 1.7320508075688772f;
            float *so = sh_out + (size_t)e * p.sh_dim;
            so[0] = 1.f; so[1] = s3 * x; so[2] = s3 * y; so[3] = s3 * z;
            if (p.sh_dim == 9) {
                const float s5 = 2.23606797749979f;
                so[4] = s5 * s3 * x * z;
                so[5] = s5 * s3 * x * y;
                so[6] = s5 * (y * y - 0.5f * (x * x + z * z));
                so[7] = s5 * s3 * y * z;
                so[8] = s5 * (s3 * 0.5f) * (z * z - x * x);
            }
            g = graph_of_a ? graph_of_a[a] : a;
        }
        s_d[tid] = d;
        s_g[tid] = g;
    }
    __syncthreads();
    for (int i = tid; i < p.n_rbf * kEE; i += kEEThreads) {
        const int k = i / kEE, el = i % kEE;
        const float t = s_d[el] - p.rbf_offset[k];
        s_in[i] = expf(p.rbf_coeff * (t * t));
    }
    for (int i = tid; i < p.n_pre * kEE; i += kEEThreads) {
        const int k = i / kEE, el = i % kEE;
        const int e = e0 + el;
        s_in[p.n_rbf * kEE + i] = (pre != nullptr && e < n_pre_rows) ? pre[(size_t)e * p.n_pre + k] : 0.f;
    }
    __syncthreads();
    const int o = tid & 63, half = tid >> 6;  // 16 edges per half
    float acc[16];
    if (o < p.ns) {
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const int el = half * 16 + i;
            acc[i] = (u != nullptr) ? u[(size_t)s_g[el] * p.ns + o] : p.b1[o];
        }
        for (int k = 0; k < p.n_rbf; ++k) {
            const float w = __ldg(p.w_rbf + (size_t)k * p.ns + o);
            const float4 *v = reinterpret_cast<const float4 *>(s_in + k * kEE + half * 16);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const float4 f = v[q];
                acc[4 * q] = fmaf(w, f.x, acc[4 * q]); acc[4 * q + 1] = fmaf(w, f.y, acc[4 * q + 1]);
                acc[4 * q + 2] = fmaf(w, f.z, acc[4 * q + 2]); acc[4 * q + 3] = fmaf(w, f.w, acc[4 * q + 3]);
            }
        }
        for (int k = 0; k < p.n_pre; ++k) {
            const float w = __ldg(p.w_pre + (size_t)k * p.ns + o);
            const float *v = s_in + (p.n_rbf + k) * kEE + half * 16;
#pragma unroll
            for (int i = 0; i < 16; ++i) acc[i] = fmaf(w, v[i], acc[i]);
        }
#pragma unroll
        for (int i = 0; i < 16; ++i) s_r[o * kEE + half * 16 + i] = fmaxf(acc[i], 0.f);
        if (p.w2 == nullptr) {
            // folded form: the second Linear lives in the consuming convolution's W1, emit the hidden activations
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const int e = e0 + half * 16 + i;
                if (e < n_edges) emb[(size_t)e * p.ns + o] = fmaxf(acc[i], 0.f);
            }
        }
    }
    if (p.w2 == nullptr) return;
    __syncthreads();
    if (o < p.ns) {
#pragma unroll
        for (int i = 0; i < 16; ++i) acc[i] = p.b2[o];
        for (int k = 0; k < p.ns; ++k) {
            const float w = __ldg(p.w2 + (size_t)k * p.ns + o);
            const float4 *v = reinterpret_cast<const float4 *>(s_r + k * kEE + half * 16);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const float4 f = v[q];
                acc[4 * q] = fmaf(w, f.x, acc[4 * q]); acc[4 * q + 1] = fmaf(w, f.y, acc[4 * q + 1]);
                acc[4 * q + 2] = fmaf(w, f.z, acc[4 * q + 2]); acc[4 * q + 3] = fmaf(w, f.w, acc[4 * q + 3]);
            }
        }
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const int e = e0 + half * 16 + i;
            if (e < n_edges) emb[(size_t)e * p.ns + o] = acc[i];
        }
    }
}

// Folded form (mlp.w2 == NULL, ns % 4 == 0): 64 edges per block, 128 threads = 16 output quads x 8 edge octets; every
// thread keeps a 4 x 8 register tile, so one weight float4 + two shared-memory float4 feed 32 FMAs.
constexpr int kFE = 64;
__global__ void __launch_bounds__(128)
edge_embed_fold_kernel(const float *__restrict__ pos_a, const float *__restrict__ pos_b, const int32_t *__restrict__ edge,
                       int cap, const int32_t *__restrict__ n_edges_dev, const int32_t *__restrict__ graph_of_a,
                       const float *__restrict__ pre, int n_pre_rows, const float *__restrict__ u, ddp_edge_mlp_t p,
                       float *__restrict__ sh_out, float *__restrict__ emb) {
    __shared__ __align__(16) float s_in[(kMaxRbf + kMaxPre) * kFE];   // [k][edge]
    __shared__ __align__(16) float s_w[(kMaxRbf + kMaxPre) * kMaxNs]; // [k][ns] first-layer weights (rbf rows, then pre rows)
    __shared__ float s_d[kFE];
    __shared__ int s_g[kFE];
    const int n_edges = min(*n_edges_dev, cap);
    const int e0 = blockIdx.x * kFE;
    if (e0 >= n_edges) return;
    const int tid = threadIdx.x;
    // stage the weights once per block (coalesced; the K loop below then runs out of shared memory instead of paying an
    // L2 round trip per unrolled group), overlapping the dependent edge -> position loads of the geometry phase
    {
        const int n4r = p.n_rbf * p.ns / 4, n4p = p.n_pre * p.ns / 4;
        for (int i = tid; i < n4r; i += 128) reinterpret_cast<float4 *>(s_w)[i] = __ldg(reinterpret_cast<const float4 *>(p.w_rbf) + i);
        for (int i = tid; i < n4p; i += 128) reinterpret_cast<float4 *>(s_w)[n4r + i] = __ldg(reinterpret_cast<const float4 *>(p.w_pre) + i);
    }
    if (tid < kFE) {
        const int e = e0 + tid;
        float d = 0.f;
        int g = 0;
        if (e < n_edges) {
            const int a = edge[e], b = edge[cap + e];
            const float vx = pos_b[3 * b] - pos_a[3 * a], vy = pos_b[3 * b + 1] - pos_a[3 * a + 1],
                        vz = pos_b[3 * b + 2] - pos_a[3 * a + 2];
            d = sqrtf(vx * vx + vy * vy + vz * vz);
            const float inv = 1.f / fmaxf(d, 1e-12f);
            const float x = vx * inv, y = vy * inv, z = vz * inv;
            const float s3 = 1.7320508075688772f;
            float *so = sh_out + (size_t)e * p.sh_dim;
            so[0] = 1.f; so[1] = s3 * x; so[2] = s3 * y; so[3] = s3 * z;
            if (p.sh_dim == 9) {
                const float s5 = 2.23606797749979f;
                so[4] = s5 * s3 * x * z;
                so[5] = s5 * s3 * x * y;
                so[6] = s5 * (y * y - 0.5f * (x * x + z * z));
                so[7] = s5 * s3 * y * z;
                so[8] = s5 * (s3 * 0.5f) * (z * z - x * x);
            }
            g = graph_of_a ? graph_of_a[a] : a;
        }
        s_d[tid] = d;
        s_g[tid] = g;
    }
    __syncthreads();
    for (int i = tid; i < p.n_rbf * kFE; i += 128) {
        const int k = i / kFE, el = i % kFE;
        const float t = s_d[el] - p.rbf_offset[k];
        s_in[i] = expf(p.rbf_coeff * (t * t));
    }
    for (int i = tid; i < p.n_pre * kFE; i += 128) {
        const int k = i / kFE, el = i % kFE;
        const int e = e0 + el;
        s_in[p.n_rbf * kFE + i] = (pre != nullptr && e < n_pre_rows) ? pre[(size_t)e * p.n_pre + k] : 0.f;
    }
    __syncthreads();
    const int quad = tid & 15, oct = tid >> 4;
    const int o = 4 * quad;
    if (o >= p.ns) return;
    float acc[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const float4 b = (u != nullptr) ? *reinterpret_cast<const float4 *>(u + (size_t)s_g[oct * 8 + i] * p.ns + o)
                                        : *reinterpret_cast<const float4 *>(p.b1 + o);
        acc[i][0] = b.x; acc[i][1] = b.y; acc[i][2] = b.z; acc[i][3] = b.w;
    }
    const int n_k = p.n_rbf + p.n_pre;
#pragma unroll 8
    for (int k = 0; k < n_k; ++k) {
        const float4 w = *reinterpret_cast<const float4 *>(s_w + k * p.ns + o);
        const float4 v0 = *reinterpret_cast<const float4 *>(s_in + k * kFE + oct * 8);
        const float4 v1 = *reinterpret_cast<const float4 *>(s_in + k * kFE + oct * 8 + 4);
        const float v[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            acc[i][0] = fmaf(w.x, v[i], acc[i][0]); acc[i][1] = fmaf(w.y, v[i], acc[i][1]);
            acc[i][2] = fmaf(w.z, v[i], acc[i][2]); acc[i][3] = fmaf(w.w, v[i], acc[i][3]);
        }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int e = e0 + oct * 8 + i;
        if (e < n_edges)
            *reinterpret_cast<float4 *>(emb + (size_t)e * p.ns + o) =
                make_float4(fmaxf(acc[i][0], 0.f), fmaxf(acc[i][1], 0.f), fmaxf(acc[i][2], 0.f), fmaxf(acc[i][3], 0.f));
    }
}

// ---------------------------------------------------------------------------------------------
constexpr int kMaxUpdates = 4;
struct UpdatePack { ddp_update_t u[kMaxUpdates]; int n; };

// FIXED: the sums are int64 fixed point (ddp_node_update*_fixed, DDP_ACC_FIXED_SHIFT), converted on load.
template <bool FIXED>
__device__ __forceinline__ float load_sum(const float *sum, size_t off) {
    if (FIXED) return ddp_from_fixed(reinterpret_cast<const long long *>(sum)[off]);
    return sum[off];
}
template <bool FIXED>
__device__ __forceinline__ float2 load_sum2(const float *sum, size_t off) {
    if (FIXED) {
        const long long *q = reinterpret_cast<const long long *>(sum) + off;
        return make_float2(ddp_from_fixed(q[0]), ddp_from_fixed(q[1]));
    }
    return *reinterpret_cast<const float2 *>(sum + off);
}

// Flat float2 form: one thread per channel pair, few registers, full occupancy (f_new, strides even, 8-byte aligned bases).
template <bool FIXED>
__global__ void __launch_bounds__(256) node_update_vec_kernel(const float *__restrict__ old_x, int f_old, int ld_old, UpdatePack up,
                                                              int n, int f_new, float *__restrict__ new_x, int ld_new) {
    const int h = f_new >> 1;
    const int total = n * h;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
        const int node = idx / h, c = 2 * (idx - node * h);
        float2 v = make_float2(0.f, 0.f);
        if (old_x != nullptr && c < f_old) v = *reinterpret_cast<const float2 *>(old_x + (size_t)node * ld_old + c);
#pragma unroll
        for (int k = 0; k < kMaxUpdates; ++k) {
            if (k < up.n && __ldg(up.u[k].n_edges_dev) > 0) {
                float2 m = make_float2(0.f, 0.f);
                if (up.u[k].sum != nullptr) {
                    m = load_sum2<FIXED>(up.u[k].sum, (size_t)node * f_new + c);
                    if (up.u[k].deg != nullptr) {
                        const int dg = __ldg(up.u[k].deg + node);
                        const float cnt = (float)(dg < 1 ? 1 : dg);
                        m.x = __fdiv_rn(m.x, cnt);
                        m.y = __fdiv_rn(m.y, cnt);
                    }
                }
                float2 sc = make_float2(1.f, 1.f), sf = make_float2(0.f, 0.f);
                if (up.u[k].scale != nullptr && up.u[k].deg != nullptr) sc = __ldg(reinterpret_cast<const float2 *>(up.u[k].scale + c));
                if (up.u[k].shift != nullptr) sf = __ldg(reinterpret_cast<const float2 *>(up.u[k].shift + c));
                v.x += fmaf(m.x, sc.x, sf.x);
                v.y += fmaf(m.y, sc.y, sf.y);
            }
        }
        *reinterpret_cast<float2 *>(new_x + (size_t)node * ld_new + c) = v;
    }
}

// Up to three node types (ligand / atom / receptor) of one interaction layer in one launch: blockIdx.y selects the job.
constexpr int kMaxNodeJobs = 3;
struct NodeJobs { ddp_node_update_job_t j[kMaxNodeJobs]; };
constexpr int kNodesPerThread = 4;
template <bool FIXED>
__global__ void __launch_bounds__(256) node_update_multi_kernel(NodeJobs jobs) {
    // one thread = one channel pair of kNodesPerThread consecutive nodes: the per-channel scale / shift and the live
    // flags are loaded once, the node rows (old features, sums) are issued together before the arithmetic
    const ddp_node_update_job_t &J = jobs.j[blockIdx.y];
    const int h = J.f_new >> 1;
    const int groups = (J.n + kNodesPerThread - 1) / kNodesPerThread;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= groups * h) return;
    const int g = idx / h, c = 2 * (idx - g * h);
    float2 sc[4], shift = make_float2(0.f, 0.f);
    bool has_sum[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        has_sum[k] = false;
        sc[k] = make_float2(1.f, 1.f);
        if (k < J.n_updates && __ldg(J.updates[k].n_edges_dev) > 0) {
            const ddp_update_t &u = J.updates[k];
            has_sum[k] = u.sum != nullptr;
            if (u.scale != nullptr && u.deg != nullptr) sc[k] = __ldg(reinterpret_cast<const float2 *>(u.scale + c));
            if (u.shift != nullptr) {
                const float2 sf = __ldg(reinterpret_cast<const float2 *>(u.shift + c));
                shift.x += sf.x; shift.y += sf.y;
            }
        }
    }
    const int node0 = g * kNodesPerThread;
    float2 v[kNodesPerThread], m[4][kNodesPerThread];
#pragma unroll
    for (int i = 0; i < kNodesPerThread; ++i) {
        const int node = node0 + i;
        v[i] = make_float2(0.f, 0.f);
        if (node < J.n && J.old_x != nullptr && c < J.f_old) v[i] = *reinterpret_cast<const float2 *>(J.old_x + (size_t)node * J.ld_old + c);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            m[k][i] = make_float2(0.f, 0.f);
            if (has_sum[k] && node < J.n) m[k][i] = load_sum2<FIXED>(J.updates[k].sum, (size_t)node * J.f_new + c);
        }
    }
#pragma unroll
    for (int i = 0; i < kNodesPerThread; ++i) {
        const int node = node0 + i;
        if (node >= J.n) break;
        float2 r = v[i];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (has_sum[k]) {
                float2 mm = m[k][i];
                if (J.updates[k].deg != nullptr) {
                    const int dg = __ldg(J.updates[k].deg + node);
                    const float cnt = (float)(dg < 1 ? 1 : dg);
                    mm.x = __fdiv_rn(mm.x, cnt);
                    mm.y = __fdiv_rn(mm.y, cnt);
                }
                r.x = fmaf(mm.x, sc[k].x, r.x);
                r.y = fmaf(mm.y, sc[k].y, r.y);
            }
        }
        r.x += shift.x; r.y += shift.y;
        *reinterpret_cast<float2 *>(J.new_x + (size_t)node * J.ld_new + c) = r;
    }
}

template <bool FIXED>
__global__ void node_update_kernel(const float *__restrict__ old_x, int f_old, int ld_old, UpdatePack up, int n,
                                   int f_new, float *__restrict__ new_x, int ld_new) {
    const int lane = threadIdx.x & 31;
    const int warps = (gridDim.x * blockDim.x) >> 5;
    bool live[kMaxUpdates];
#pragma unroll
    for (int k = 0; k < kMaxUpdates; ++k) live[k] = k < up.n && *up.u[k].n_edges_dev > 0;
    for (int node = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; node < n; node += warps) {
        float cnt[kMaxUpdates];
#pragma unroll
        for (int k = 0; k < kMaxUpdates; ++k) {
            cnt[k] = 1.f;
            if (live[k] && up.u[k].deg != nullptr) {
                const int dg = up.u[k].deg[node];
                cnt[k] = (float)(dg < 1 ? 1 : dg);
            }
        }
        for (int c = lane; c < f_new; c += 32) {
            float v = (old_x != nullptr && c < f_old) ? old_x[(size_t)node * ld_old + c] : 0.f;
#pragma unroll
            for (int k = 0; k < kMaxUpdates; ++k) {
                if (live[k]) {
                    const float m = up.u[k].sum ? __fdiv_rn(load_sum<FIXED>(up.u[k].sum, (size_t)node * f_new + c), cnt[k]) : 0.f;
                    const float sc = (up.u[k].scale && up.u[k].deg) ? __ldg(up.u[k].scale + c) : 1.f;
                    const float sf = up.u[k].shift ? __ldg(up.u[k].shift + c) : 0.f;
                    v += fmaf(m, sc, sf);
                }
            }
            new_x[(size_t)node * ld_new + c] = v;
        }
    }
}

// ---------------------------------------------------------------------------------------------
__global__ void segment_mean_kernel(const float *__restrict__ src, const int32_t *__restrict__ idx,
                                    const int32_t *__restrict__ ptr, int n_seg, int width, int ld,
                                    float *__restrict__ out, int ld_out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_seg * width) return;
    const int g = i / width, c = i % width;
    float s = 0.f;
    const int beg = ptr[g], end = ptr[g + 1];
    for (int r = beg; r < end; ++r) s += src[(size_t)(idx ? idx[r] : r) * ld + c];
    const int cnt = end - beg;
    out[(size_t)g * ld_out + c] = s / (float)(cnt < 1 ? 1 : cnt);
}

__global__ void bond_geometry_kernel(const float *__restrict__ pos, const int32_t *__restrict__ bonds, int n_bonds,
                                     const float *__restrict__ x, int ldx, int ns, float *__restrict__ mid,
                                     float *__restrict__ y2, float *__restrict__ attr) {
    const int bnd = blockIdx.x;
    if (bnd >= n_bonds) return;
    const int b0 = bonds[bnd], b1 = bonds[n_bonds + bnd];
    if (threadIdx.x == 0) {
        const float ax = pos[3 * b0], ay = pos[3 * b0 + 1], az = pos[3 * b0 + 2];
        const float bx = pos[3 * b1], by = pos[3 * b1 + 1], bz = pos[3 * b1 + 2];
        mid[3 * bnd] = (ax + bx) / 2.f; mid[3 * bnd + 1] = (ay + by) / 2.f; mid[3 * bnd + 2] = (az + bz) / 2.f;
        const float vx = bx - ax, vy = by - ay, vz = bz - az;
        const float inv = 1.f / fmaxf(sqrtf(vx * vx + vy * vy + vz * vz), 1e-12f);
        const float X = vx * inv, Y = vy * inv, Z = vz * inv;
        const float s3 = 1.7320508075688772f, s5 = 2.23606797749979f;
        y2[5 * bnd + 0] = s5 * s3 * X * Z;
        y2[5 * bnd + 1] = s5 * s3 * X * Y;
        y2[5 * bnd + 2] = s5 * (Y * Y - 0.5f * (X * X + Z * Z));
        y2[5 * bnd + 3] = s5 * s3 * Y * Z;
        y2[5 * bnd + 4] = s5 * (s3 * 0.5f) * (Z * Z - X * X);
    }
    for (int c = threadIdx.x; c < ns; c += blockDim.x) attr[(size_t)bnd * ns + c] = x[(size_t)b0 * ldx + c] + x[(size_t)b1 * ldx + c];
}

__global__ void tor_edge_sh_kernel(const float *__restrict__ sh, int sh_dim, const float *__restrict__ y2,
                                   const float *__restrict__ c121, const int32_t *__restrict__ edge,
                                   const int32_t *__restrict__ n_edges_dev, int cap, float *__restrict__ sh_tor) {
    __shared__ float sc[45];
    for (int i = threadIdx.x; i < 45; i += blockDim.x) sc[i] = c121[i];
    __syncthreads();
    const int n_edges = min(*n_edges_dev, cap);
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n_edges; e += gridDim.x * blockDim.x) {
        const int bnd = edge[e];
        float a[3] = {sh[(size_t)e * sh_dim + 1], sh[(size_t)e * sh_dim + 2], sh[(size_t)e * sh_dim + 3]};
        float o[3] = {0.f, 0.f, 0.f};
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < 5; ++j) {
                const float ab = a[i] * y2[5 * bnd + j];
#pragma unroll
                for (int k = 0; k < 3; ++k) o[k] = fmaf(sc[(i * 5 + j) * 3 + k], ab, o[k]);
            }
        *reinterpret_cast<float4 *>(sh_tor + 4 * (size_t)e) = make_float4(1.f, o[0], o[1], o[2]);
    }
}

// Generic form: out[e][p.out_off + k] = sum_{i, j} ctab[p.c_off + (i * 5 + j) * p.d_out + k] * sh[e][p.in_off + i] * y2[bond][j]
constexpr int kMaxFtpPaths = 8;
struct FtpPack { ddp_ftp_path_t p[kMaxFtpPaths]; int n; };

__global__ void tor_edge_sh_generic_kernel(const float *__restrict__ sh, int sh_dim, const float *__restrict__ y2, FtpPack fp,
                                           const float *__restrict__ ctab, const int32_t *__restrict__ edge,
                                           const int32_t *__restrict__ n_edges_dev, int cap, float *__restrict__ out, int out_dim) {
    const int n_edges = min(*n_edges_dev, cap);
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n_edges; e += gridDim.x * blockDim.x) {
        const int bnd = edge[e];
        float y[5];
#pragma unroll
        for (int j = 0; j < 5; ++j) y[j] = y2[5 * bnd + j];
        for (int q = 0; q < fp.n; ++q) {
            const ddp_ftp_path_t p = fp.p[q];
            for (int k = 0; k < p.d_out; ++k) {
                float o = 0.f;
                for (int i = 0; i < p.d_in; ++i) {
                    const float a = sh[(size_t)e * sh_dim + p.in_off + i];
#pragma unroll
                    for (int j = 0; j < 5; ++j) o = fmaf(__ldg(ctab + p.c_off + (i * 5 + j) * p.d_out + k), a * y[j], o);
                }
                out[(size_t)e * out_dim + p.out_off + k] = o;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
constexpr int kMaxLayers = 4;
struct MlpPack { ddp_mlp_layer_t l[kMaxLayers]; int n; };

__global__ void row_mlp_kernel(const float *__restrict__ in, int n, int ld_in, MlpPack mp,
                               const float *__restrict__ row_scale, float *__restrict__ out, int ld_out) {
    __shared__ float buf[2][256];
    __shared__ float red[8];
    const int row = blockIdx.x;
    if (row >= n) return;
    for (int k = threadIdx.x; k < mp.l[0].n_in; k += blockDim.x) buf[0][k] = in[(size_t)row * ld_in + k];
    __syncthreads();
    int cur = 0;
    for (int l = 0; l < mp.n; ++l) {
        const ddp_mlp_layer_t L = mp.l[l];
        if (L.n_out == 1) {
            // single output: the threads split K and reduce (a lone thread would chain n_in dependent loads)
            float part = 0.f;
            for (int k = threadIdx.x; k < L.n_in; k += blockDim.x) part = fmaf(__ldg(L.wt + k), buf[cur][k], part);
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) part += __shfl_xor_sync(0xffffffffu, part, off);
            if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = part;
            __syncthreads();
            if (threadIdx.x == 0) {
                float acc = L.b ? L.b[0] : 0.f;
                for (int w = 0; w < (int)(blockDim.x >> 5); ++w) acc += red[w];
                if (L.act == 1) acc = fmaxf(acc, 0.f);
                else if (L.act == 2) acc = tanhf(acc);
                buf[cur ^ 1][0] = acc;
            }
        } else {
            for (int o = threadIdx.x; o < L.n_out; o += blockDim.x) {
                float acc = L.b ? L.b[o] : 0.f;
#pragma unroll 8
                for (int k = 0; k < L.n_in; ++k) acc = fmaf(__ldg(L.wt + (size_t)k * L.n_out + o), buf[cur][k], acc);
                if (L.act == 1) acc = fmaxf(acc, 0.f);
                else if (L.act == 2) acc = tanhf(acc);
                buf[cur ^ 1][o] = acc;
            }
        }
        __syncthreads();
        cur ^= 1;
    }
    const float sc = row_scale ? row_scale[row] : 1.f;
    for (int o = threadIdx.x; o < mp.l[mp.n - 1].n_out; o += blockDim.x) out[(size_t)row * ld_out + o] = buf[cur][o] * sc;
}

__global__ void tr_rot_head_kernel(const float *__restrict__ g, const float *__restrict__ sig, int sig_dim,
                                   const float *__restrict__ tr_w1t, const float *__restrict__ tr_b1,
                                   const float *__restrict__ tr_w2, const float *__restrict__ tr_b2,
                                   const float *__restrict__ rot_w1t, const float *__restrict__ rot_b1,
                                   const float *__restrict__ rot_w2, const float *__restrict__ rot_b2, int hid,
                                   const float *__restrict__ tr_sigma, const float *__restrict__ so3_norm,
                                   float *__restrict__ tr_out, float *__restrict__ rot_out) {
    __shared__ float red[2][128];
    const int b = blockIdx.x, j = threadIdx.x;
    const float *gg = g + 12 * (size_t)b;
    const float tx = gg[0] + gg[6], ty = gg[1] + gg[7], tz = gg[2] + gg[8];
    const float rx = gg[3] + gg[9], ry = gg[4] + gg[10], rz = gg[5] + gg[11];
    const float tn = sqrtf(tx * tx + ty * ty + tz * tz), rn = sqrtf(rx * rx + ry * ry + rz * rz);
    float ht = 0.f, hr = 0.f;
    if (j < hid) {
        float at = fmaf(tr_w1t[j], tn, tr_b1[j]), ar = fmaf(rot_w1t[j], rn, rot_b1[j]);
        for (int k = 0; k < sig_dim; ++k) {
            const float s = sig[(size_t)b * sig_dim + k];
            at = fmaf(tr_w1t[(size_t)(1 + k) * hid + j], s, at);
            ar = fmaf(rot_w1t[(size_t)(1 + k) * hid + j], s, ar);
        }
        ht = fmaxf(at, 0.f) * tr_w2[j];
        hr = fmaxf(ar, 0.f) * rot_w2[j];
    }
    red[0][j] = ht; red[1][j] = hr;
    __syncthreads();
    if (j == 0) {
        float st = tr_b2[0], sr = rot_b2[0];
        for (int k = 0; k < hid; ++k) { st += red[0][k]; sr += red[1][k]; }
        const float ft = st / tn / tr_sigma[b], fr = sr / rn * so3_norm[b];
        tr_out[3 * b] = tx * ft; tr_out[3 * b + 1] = ty * ft; tr_out[3 * b + 2] = tz * ft;
        rot_out[3 * b] = rx * fr; rot_out[3 * b + 1] = ry * fr; rot_out[3 * b + 2] = rz * fr;
    }
}

}  // namespace

static inline int grid_for(size_t total, int threads) {
    size_t g = (total + threads - 1) / threads;
    const size_t cap = (size_t)ddp_num_sms() * 8;
    return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

extern "C" int ddp_graph_sigma_proj(const float *t, int32_t n_graphs, float scale, const float *freq, int32_t sig_dim,
                                    const float *w, const float *b, int32_t n_proj, int32_t ns, float *sig, float *out,
                                    void *stream) {
    if (!t || !freq || !w || !b || !sig || !out) return DDP_E_ARG;
    if (n_graphs <= 0 || n_proj <= 0 || sig_dim <= 0 || sig_dim > 1024 || ns <= 0) return DDP_E_SHAPE;
    graph_sigma_proj_kernel<<<dim3(n_graphs, n_proj), 64, sig_dim * sizeof(float), (cudaStream_t)stream>>>(
        t, scale, freq, sig_dim, w, b, n_graphs, ns, sig, out);
    DDP_LAUNCH_CHECK();
    return 0;
}

extern "C" int ddp_node_init(const float *static_part, const float *u, const int32_t *graph_of, int32_t n, int32_t ns,
                             float *out, int32_t ld_out, void *stream) {
    if (!static_part || !u || !graph_of || !out) return DDP_E_ARG;
    if (n <= 0) return 0;
    node_init_kernel<<<grid_for((size_t)n * ns, 256), 256, 0, (cudaStream_t)stream>>>(static_part, u, graph_of, n, ns, out, ld_out);
    DDP_LAUNCH_CHECK();
    return 0;
}

extern "C" int ddp_node_static_embed(const int64_t *cat, int32_t n, int32_t n_cat, const float *table, const int32_t *table_off,
                                     const float *lm, int32_t n_lm, const float *w_emb_t, const float *w_lm_t, int32_t ns,
                                     float *out, void *stream) {
    if (!cat || !table || !table_off || !out || n_cat <= 0 || ns <= 0) return DDP_E_ARG;
    if (n_lm > 0 && (!lm || !w_lm_t)) return DDP_E_ARG;
    if (n_lm < 0 || (size_t)(ns + n_lm) * sizeof(float) > 40 * 1024) return DDP_E_SHAPE;
    if (n <= 0) return 0;
    node_static_embed_kernel<<<n, kStaticThreads, (size_t)(ns + n_lm) * sizeof(float), (cudaStream_t)stream>>>(
        cat, n_cat, table, table_off, lm, n_lm, w_emb_t, w_lm_t, ns, out);
    DDP_LAUNCH_CHECK();
    return 0;
}

extern "C" int ddp_edge_embed(const float *pos_a, const float *pos_b, const int32_t *edge, int32_t edge_cap,
                              const int32_t *n_edges_dev, const int32_t *graph_of_a, const float *pre,
                              int32_t n_pre_rows, const float *u, const ddp_edge_mlp_t *mlp, float *sh, float *emb,
                              void *stream) {
    if (!pos_a || !pos_b || !edge || !n_edges_dev || !mlp || !sh || !emb) return DDP_E_ARG;
    if (mlp->ns > kMaxNs || mlp->n_rbf > kMaxRbf || mlp->n_pre > kMaxPre || (mlp->sh_dim != 4 && mlp->sh_dim != 9))
        return DDP_E_SHAPE;
    if (!u && !mlp->b1) return DDP_E_ARG;
    if (edge_cap <= 0) return 0;
    const bool aligned = mlp->ns % 4 == 0 && reinterpret_cast<uintptr_t>(emb) % 16 == 0 && reinterpret_cast<uintptr_t>(u) % 16 == 0 &&
                         reinterpret_cast<uintptr_t>(mlp->w_rbf) % 16 == 0 && reinterpret_cast<uintptr_t>(mlp->w_pre) % 16 == 0 &&
                         reinterpret_cast<uintptr_t>(mlp->b1) % 16 == 0;
    if (mlp->w2 == nullptr && aligned)
        edge_embed_fold_kernel<<<(edge_cap + kFE - 1) / kFE, 128, 0, (cudaStream_t)stream>>>(
            pos_a, pos_b, edge, edge_cap, n_edges_dev, graph_of_a, pre, n_pre_rows, u, *mlp, sh, emb);
    else
        edge_embed_kernel<<<(edge_cap + kEE - 1) / kEE, kEEThreads, 0, (cudaStream_t)stream>>>(
            pos_a, pos_b, edge, edge_cap, n_edges_dev, graph_of_a, pre, n_pre_rows, u, *mlp, sh, emb);
    DDP_LAUNCH_CHECK();
    return 0;
}

template <bool FIXED>
static int node_update(const float *old_x, int32_t f_old, int32_t ld_old, const ddp_update_t *updates, int32_t n_updates, int32_t n,
                       int32_t f_new, float *new_x, int32_t ld_new, void *stream) {
    if (!updates || !new_x || n_updates < 0 || n_updates > kMaxUpdates) return DDP_E_ARG;
    if (n <= 0) return 0;
    UpdatePack up;
    up.n = n_updates;
    for (int i = 0; i < n_updates; ++i) up.u[i] = updates[i];
    // vector path: even widths / strides and 8-byte aligned bases (every buffer of the resident plan qualifies)
    bool vec = (f_new % 2 == 0) && (f_old % 2 == 0) && (ld_new % 2 == 0) && (ld_old % 2 == 0) && f_new <= 192 &&
               (reinterpret_cast<uintptr_t>(new_x) % 8 == 0) && (reinterpret_cast<uintptr_t>(old_x) % 8 == 0);
    for (int i = 0; i < n_updates; ++i) vec = vec && (reinterpret_cast<uintptr_t>(updates[i].sum) % 8 == 0);
    for (int i = 0; i < n_updates; ++i)
        vec = vec && (reinterpret_cast<uintptr_t>(updates[i].scale) % 8 == 0) && (reinterpret_cast<uintptr_t>(updates[i].shift) % 8 == 0);
    if (vec)
        node_update_vec_kernel<FIXED><<<(int)(((size_t)n * (f_new / 2) + 255) / 256), 256, 0, (cudaStream_t)stream>>>(old_x, f_old, ld_old, up, n,
                                                                                                      f_new, new_x, ld_new);
    else
        node_update_kernel<FIXED><<<grid_for((size_t)n * 32, 256), 256, 0, (cudaStream_t)stream>>>(old_x, f_old, ld_old, up, n, f_new, new_x, ld_new);
    DDP_LAUNCH_CHECK();
    return 0;
}

extern "C" int ddp_node_update(const float *old_x, int32_t f_old, int32_t ld_old, const ddp_update_t *updates,
                               int32_t n_updates, int32_t n, int32_t f_new, float *new_x, int32_t ld_new, void *stream) {
    return node_update<false>(old_x, f_old, ld_old, updates, n_updates, n, f_new, new_x, ld_new, stream);
}

extern "C" int ddp_node_update_fixed(const float *old_x, int32_t f_old, int32_t ld_old, const ddp_update_t *updates,
                                     int32_t n_updates, int32_t n, int32_t f_new, float *new_x, int32_t ld_new, void *stream) {
    return node_update<true>(old_x, f_old, ld_old, updates, n_updates, n, f_new, new_x, ld_new, stream);
}

template <bool FIXED>
static int node_update_multi(const ddp_node_update_job_t *jobs_host, int32_t n_jobs, void *stream) {
    if (!jobs_host || n_jobs < 0 || n_jobs > kMaxNodeJobs) return DDP_E_ARG;
    NodeJobs jobs;
    size_t most = 0;
    int m = 0;
    for (int i = 0; i < n_jobs; ++i) {
        const ddp_node_update_job_t &J = jobs_host[i];
        if (J.n <= 0) continue;
        if (!J.new_x || J.n_updates < 0 || J.n_updates > 4) return DDP_E_ARG;
        bool ok = (J.f_new % 2 == 0) && (J.f_old % 2 == 0) && (J.ld_new % 2 == 0) && (J.ld_old % 2 == 0) &&
                  (reinterpret_cast<uintptr_t>(J.new_x) % 8 == 0) && (reinterpret_cast<uintptr_t>(J.old_x) % 8 == 0);
        for (int k = 0; k < J.n_updates; ++k)
            ok = ok && J.updates[k].n_edges_dev && (reinterpret_cast<uintptr_t>(J.updates[k].sum) % 8 == 0) &&
                 (reinterpret_cast<uintptr_t>(J.updates[k].scale) % 8 == 0) && (reinterpret_cast<uintptr_t>(J.updates[k].shift) % 8 == 0);
        if (!ok) return DDP_E_UNSUPPORTED;
        jobs.j[m++] = J;
        const size_t tot = (size_t)((J.n + kNodesPerThread - 1) / kNodesPerThread) * (J.f_new / 2);
        most = tot > most ? tot : most;
    }
    if (m == 0) return 0;
    node_update_multi_kernel<FIXED><<<dim3((unsigned)((most + 255) / 256), m), 256, 0, (cudaStream_t)stream>>>(jobs);
    DDP_LAUNCH_CHECK();
    return 0;
}

extern "C" int ddp_node_update_multi(const ddp_node_update_job_t *jobs_host, int32_t n_jobs, void *stream) {
    return node_update_multi<false>(jobs_host, n_jobs, stream);
}

extern "C" int ddp_node_update_multi_fixed(const ddp_node_update_job_t *jobs_host, int32_t n_jobs, void *stream) {
    return node_update_multi<true>(jobs_host, n_jobs, stream);
}

extern "C" int ddp_segment_mean(const float *src, const int32_t *idx, const int32_t *ptr, int32_t n_seg, int32_t width,
                                int32_t ld, float *out, int32_t ld_out, void *stream) {
    if (!src || !ptr || !out) return DDP_E_ARG;
    if (n_seg <= 0 || width <= 0) return 0;
    segment_mean_kernel<<<(n_seg * width + 127) / 128, 128, 0, (cudaStream_t)stream>>>(src, idx, ptr, n_seg, width, ld, out, ld_out);
    DDP_LAUNCH_CHECK();
    return 0;
}

extern "C" int ddp_bond_geometry(const float *pos, const int32_t *bonds, int32_t n_bonds, const float *x, int32_t ldx,
                                 int32_t ns, float *mid, float *y2, float *attr, void *stream) {
    if (!pos || !bonds || !x || !mid || !y2 || !attr) return DDP_E_ARG;
    if (n_bonds <= 0) return 0;
    bond_geometry_kernel<<<n_bonds, 64, 0, (cudaStream_t)stream>>>(pos, bonds, n_bonds, x, ldx, ns, mid, y2, attr);
    DDP_LAUNCH_CHECK();
    return 0;
}

extern "C" int ddp_tor_edge_sh(const float *sh, int32_t sh_dim, const float *y2, const float *c121, const int32_t *edge,
                               const int32_t *n_edges_dev, int32_t edge_cap, float *sh_tor, void *stream) {
    if (!sh || !y2 || !c121 || !edge || !n_edges_dev || !sh_tor) return DDP_E_ARG;
    if (edge_cap <= 0) return 0;
    tor_edge_sh_kernel<<<grid_for(edge_cap, 128), 128, 0, (cudaStream_t)stream>>>(sh, sh_dim, y2, c121, edge, n_edges_dev,
                                                                                 edge_cap, sh_tor);
    DDP_LAUNCH_CHECK();
    return 0;
}

extern "C" int ddp_tor_edge_sh_generic(const float *sh, int32_t sh_dim, const float *y2, const ddp_ftp_path_t *paths_host,
                                       int32_t n_paths, const float *ctab, const int32_t *edge, const int32_t *n_edges_dev,
                                       int32_t edge_cap, float *out, int32_t out_dim, void *stream) {
    if (!sh || !y2 || !paths_host || !ctab || !edge || !n_edges_dev || !out) return DDP_E_ARG;
    if (n_paths <= 0 || n_paths > kMaxFtpPaths) return DDP_E_SHAPE;
    FtpPack fp;
    fp.n = n_paths;
    for (int i = 0; i < n_paths; ++i) {
        fp.p[i] = paths_host[i];
        if (fp.p[i].in_off < 0 || fp.p[i].in_off + fp.p[i].d_in > sh_dim || fp.p[i].out_off < 0 || fp.p[i].out_off + fp.p[i].d_out > out_dim)
            return DDP_E_SHAPE;
    }
    if (edge_cap <= 0) return 0;
    tor_edge_sh_generic_kernel<<<grid_for(edge_cap, 128), 128, 0, (cudaStream_t)stream>>>(sh, sh_dim, y2, fp, ctab, edge, n_edges_dev,
                                                                                         edge_cap, out, out_dim);
    DDP_LAUNCH_CHECK();
    return 0;
}

extern "C" int ddp_row_mlp(const float *in, int32_t n, int32_t ld_in, const ddp_mlp_layer_t *layers_host, int32_t n_layers,
                           const float *row_scale, float *out, int32_t ld_out, void *stream) {
    if (!in || !layers_host || !out || n_layers <= 0 || n_layers > kMaxLayers) return DDP_E_ARG;
    MlpPack mp;
    mp.n = n_layers;
    for (int i = 0; i < n_layers; ++i) {
        mp.l[i] = layers_host[i];
        if (mp.l[i].n_in > 256 || mp.l[i].n_out > 256 || !mp.l[i].wt) return DDP_E_SHAPE;
    }
    if (n <= 0) return 0;
    row_mlp_kernel<<<n, 64, 0, (cudaStream_t)stream>>>(in, n, ld_in, mp, row_scale, out, ld_out);
    DDP_LAUNCH_CHECK();
    return 0;
}

extern "C" int ddp_tr_rot_head(const float *g, const float *sig, int32_t sig_dim, int32_t n_graphs, const float *tr_w1t,
                               const float *tr_b1, const float *tr_w2, const float *tr_b2, const float *rot_w1t,
                               const float *rot_b1, const float *rot_w2, const float *rot_b2, int32_t hid,
                               const float *tr_sigma, const float *so3_norm, float *tr_out, float *rot_out, void *stream) {
    if (!g || !sig || !tr_w1t || !rot_w1t || !tr_out || !rot_out || !tr_sigma || !so3_norm) return DDP_E_ARG;
    if (hid > 128 || hid <= 0) return DDP_E_SHAPE;
    if (n_graphs <= 0) return 0;
    tr_rot_head_kernel<<<n_graphs, 128, 0, (cudaStream_t)stream>>>(g, sig, sig_dim, tr_w1t, tr_b1, tr_w2, tr_b2, rot_w1t, rot_b1,
                                                                 rot_w2, rot_b2, hid, tr_sigma, so3_norm, tr_out, rot_out);
    DDP_LAUNCH_CHECK();
    return 0;
}
