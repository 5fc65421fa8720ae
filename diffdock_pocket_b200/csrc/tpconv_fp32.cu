// fp32 CUDA-core tensor-product convolution (exact-arithmetic mode / generic-irreps fallback).
// One CTA = 32 edges.  The per-edge weight vector w = W2 relu(W1 a + b1) + b2 exists only as an
// 8-edge register tile per weight column; it is contracted with the table-driven Clebsch-Gordan
// basis immediately and accumulated in shared memory, then scattered with red.global.add.
// FIXED (deterministic mode, ddp_tpconv_fp32_fixed): the shared-memory tile and the global sums are int64 fixed point
// (DDP_ACC_FIXED_SHIFT), so neither the order of the warps' shared atomics nor that of the CTAs' global ones shows in
// the result.
#include "ddp_common.cuh"

namespace {

constexpr int NT = 256;
constexpr int EG = 8;         // edges per register tile
// TE edges per tile (32, or 8 for small edge sets so that a few hundred edges still spread over the SMs);
// LDS_E = TE + 4: padded edge stride (multiple of 4 for float4 reads)

struct Smem {
    float *a, *h, *x, *sh, *out, *ctab;
    int *agg;
};

template <int TE, bool FIXED>
__device__ __forceinline__ Smem carve(float *base, const ddp_tpconv_t &c, int ctab_len) {
    constexpr int LDS_E = TE + 4;
    Smem s;
    s.a = base;
    s.h = s.a + c.k1 * LDS_E;
    s.x = s.h + c.hid * LDS_E;
    s.sh = s.x + c.f_in * LDS_E;
    s.out = s.sh + c.sh_dim * LDS_E;
    s.ctab = s.out + c.f_out * LDS_E * (FIXED ? 2 : 1);     // (FIXED: int64 tile, 8-byte aligned: every stride above is even)
    s.agg = reinterpret_cast<int *>(s.ctab + ctab_len);
    return s;
}

template <int TE, bool FIXED>
__global__ void __launch_bounds__(NT, 2)
tpconv_fp32_kernel(ddp_tpconv_t c, ddp_tpconv_edges_t ed, int ctab_len, float *__restrict__ sum, uint32_t *status) {
    constexpr int LDS_E = TE + 4;
    constexpr int NEG = TE / EG;          // edge groups per tile
    constexpr int TPG = NT / NEG;         // threads per edge group in the weight-column phase
    extern __shared__ __align__(16) float smem[];
    Smem s = carve<TE, FIXED>(smem, c, ctab_len);
    unsigned long long *out_q = reinterpret_cast<unsigned long long *>(s.out);     // FIXED only
    const int tid = threadIdx.x;
    const int n_edges = min(*ed.n_edges_dev, ed.edge_cap);
    for (int i = tid; i < ctab_len; i += NT) s.ctab[i] = c.ctab[i];

    for (int tile = blockIdx.x; tile * TE < n_edges; tile += gridDim.x) {
        const int e0 = tile * TE;
        __syncthreads();
        // ---- stage edge attributes [k][e], gathered features [c][e], sh [j][e] -----------------
        for (int idx = tid; idx < TE * c.k1; idx += NT) {
            const int el = idx / c.k1, k = idx % c.k1, e = e0 + el;
            float v = 0.f;
            if (e < n_edges) {
                if (k < c.n_emb) v = ed.emb[(size_t)e * c.n_emb + k];
                else if (k < c.n_emb + c.ns && ed.p1 != nullptr) v = ed.p1[(size_t)ed.i1[e] * ed.ld1 + (k - c.n_emb)];
                else {
                    const int kk = k - c.n_emb - (ed.p1 != nullptr ? c.ns : 0);
                    v = ed.p2[(size_t)ed.i2[e] * ed.ld2 + kk];
                }
            }
            s.a[k * LDS_E + el] = v;
        }
        for (int idx = tid; idx < TE * c.f_in; idx += NT) {
            const int el = idx / c.f_in, k = idx % c.f_in, e = e0 + el;
            s.x[k * LDS_E + el] = (e < n_edges) ? ed.x[(size_t)ed.gather[e] * ed.ldx + k] : 0.f;
        }
        for (int idx = tid; idx < TE * c.sh_dim; idx += NT) {
            const int el = idx / c.sh_dim, k = idx % c.sh_dim, e = e0 + el;
            s.sh[k * LDS_E + el] = (e < n_edges) ? ed.sh[(size_t)e * c.sh_dim + k] : 0.f;
        }
        if (FIXED)
            for (int idx = tid; idx < c.f_out * LDS_E; idx += NT) out_q[idx] = 0ull;
        else
            for (int idx = tid; idx < c.f_out * LDS_E; idx += NT) s.out[idx] = 0.f;
        if (tid < TE) s.agg[tid] = (e0 + tid < n_edges) ? ed.agg[e0 + tid] : -1;
        __syncthreads();

        // ---- h = relu(W1 a + b1): unit = (hidden j, edge group) ---------------------------------
        for (int unit = tid; unit < c.hid * (TE / EG); unit += NT) {
            const int j = unit % c.hid, eg = unit / c.hid;
            float acc[EG];
            const float bj = c.b1[j];
#pragma unroll
            for (int i = 0; i < EG; ++i) acc[i] = bj;
            const float *ap = s.a + eg * EG;
#pragma unroll 8
            for (int k = 0; k < c.k1; ++k) {
                const float w = __ldg(c.w1t + (size_t)k * c.hid + j);
                const float4 v0 = *reinterpret_cast<const float4 *>(ap + k * LDS_E);
                const float4 v1 = *reinterpret_cast<const float4 *>(ap + k * LDS_E + 4);
                acc[0] = fmaf(w, v0.x, acc[0]); acc[1] = fmaf(w, v0.y, acc[1]); acc[2] = fmaf(w, v0.z, acc[2]);
                acc[3] = fmaf(w, v0.w, acc[3]); acc[4] = fmaf(w, v1.x, acc[4]); acc[5] = fmaf(w, v1.y, acc[5]);
                acc[6] = fmaf(w, v1.z, acc[6]); acc[7] = fmaf(w, v1.w, acc[7]);
            }
#pragma unroll
            for (int i = 0; i < EG; ++i) s.h[j * LDS_E + eg * EG + i] = fmaxf(acc[i], 0.f);
        }
        __syncthreads();

        // ---- weight columns: TPG consecutive columns x NEG edge groups per pass ---------------------
        const int eg = tid / TPG;
        const float *hp = s.h + eg * EG;
        // warp-uniform trip count (lanes past the last column idle but still take part in the shuffles below)
        for (int cb = (tid % TPG) & ~31; cb < c.w_numel; cb += TPG) {
            const bool active = cb + (tid & 31) < c.w_numel;
            const int col = active ? cb + (tid & 31) : c.w_numel - 1;
            float acc[EG];
            const float bc = c.b2[col];
#pragma unroll
            for (int i = 0; i < EG; ++i) acc[i] = bc;
            const float *wp = c.w2t + col;
#pragma unroll 8
            for (int k = 0; k < c.hid; ++k) {
                const float w = __ldg(wp + (size_t)k * c.w_numel);
                const float4 v0 = *reinterpret_cast<const float4 *>(hp + k * LDS_E);
                const float4 v1 = *reinterpret_cast<const float4 *>(hp + k * LDS_E + 4);
                acc[0] = fmaf(w, v0.x, acc[0]); acc[1] = fmaf(w, v0.y, acc[1]); acc[2] = fmaf(w, v0.z, acc[2]);
                acc[3] = fmaf(w, v0.w, acc[3]); acc[4] = fmaf(w, v1.x, acc[4]); acc[5] = fmaf(w, v1.y, acc[5]);
                acc[6] = fmaf(w, v1.z, acc[6]); acc[7] = fmaf(w, v1.w, acc[7]);
            }
            const int gi = c.col_group[col];
            const ddp_tp_group_t g = c.groups[gi];
            // warp-uniform: every lane active on a column of the same group, group start aligned to the warp's 32 columns
            const int gi0 = __shfl_sync(0xffffffffu, gi, 0);
            const bool same = __all_sync(0xffffffffu, active && gi == gi0);
            const bool warp_reduce = same && (g.mul_out & (g.mul_out - 1)) == 0 && g.mul_out <= 16 && ((cb - g.w_off) % g.mul_out) == 0;
            const int u = (col - g.w_off) / g.mul_out, o = (col - g.w_off) % g.mul_out;
            const float *cg = s.ctab + g.c_off;
            const float *xp = s.x + (g.x_off + u * g.d1) * LDS_E + eg * EG;
            const float *sp = s.sh + g.sh_off * LDS_E + eg * EG;
            float *op = s.out + (g.out_off + o * g.d_out) * LDS_E + eg * EG;
            for (int kk = 0; kk < g.d_out; ++kk) {
                float b[EG];
#pragma unroll
                for (int i = 0; i < EG; ++i) b[i] = 0.f;
                for (int ii = 0; ii < g.d1; ++ii)
                    for (int jj = 0; jj < g.d2; ++jj) {
                        const float cc = cg[(ii * g.d2 + jj) * g.d_out + kk];
                        if (cc != 0.f) {
#pragma unroll
                            for (int i = 0; i < EG; ++i) b[i] = fmaf(cc * xp[ii * LDS_E + i], sp[jj * LDS_E + i], b[i]);
                        }
                    }
                if (warp_reduce) {
                    // all 32 lanes hold columns of one group whose mul_out divides 32: lanes l, l + mul_out, ... feed
                    // the same output channel, so they are summed by shuffles and only mul_out lanes touch shared memory
#pragma unroll
                    for (int i = 0; i < EG; ++i) {
                        float v = acc[i] * b[i];
                        for (int off = 16; off >= g.mul_out; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
                        if ((tid & 31) < g.mul_out) {
                            if (FIXED) atomicAdd(out_q + (op - s.out) + kk * LDS_E + i, ddp_to_fixed(v, status));
                            else atomicAdd(op + kk * LDS_E + i, v);
                        }
                    }
                } else if (active) {
#pragma unroll
                    for (int i = 0; i < EG; ++i) {
                        if (FIXED) atomicAdd(out_q + (op - s.out) + kk * LDS_E + i, ddp_to_fixed(acc[i] * b[i], status));
                        else atomicAdd(op + kk * LDS_E + i, acc[i] * b[i]);
                    }
                }
            }
        }
        __syncthreads();

        // ---- scatter-add to the aggregation nodes ----------------------------------------------------
        for (int idx = tid; idx < TE * c.f_out; idx += NT) {
            const int el = idx / c.f_out, k = idx % c.f_out;
            const int node = s.agg[el];
            if (node >= 0) {
                float v = FIXED ? ddp_from_fixed((long long)out_q[k * LDS_E + el]) : s.out[k * LDS_E + el];
                if (ed.ew != nullptr) v *= ed.ew[e0 + el];
                if (ed.out_scale != nullptr) v *= ed.out_scale[k];
                if (ed.agg_deg != nullptr) v *= __frcp_rn((float)max(ed.agg_deg[node], 1));
                if (FIXED) atomicAdd(reinterpret_cast<unsigned long long *>(sum) + (size_t)node * c.f_out + k, ddp_to_fixed(v, status));
                else atomicAdd(sum + (size_t)node * c.f_out + k, v);
            }
        }
    }
}

}  // namespace

template <bool FIXED>
static int tpconv_fp32(const ddp_tpconv_t *conv, const ddp_tpconv_edges_t *edges, float *sum, uint32_t *status, void *stream) {
    if (!conv || !edges || !sum || (FIXED && !status)) return DDP_E_ARG;
    const ddp_tpconv_t &c = *conv;
    const ddp_tpconv_edges_t &e = *edges;
    if (!c.w1t || !c.b1 || !c.w2t || !c.b2 || !c.groups || !c.ctab || !c.col_group) return DDP_E_ARG;
    if (!e.emb || !e.x || !e.gather || !e.sh || !e.agg || !e.n_edges_dev) return DDP_E_ARG;
    const int parts = (e.p1 != nullptr) + (e.p2 != nullptr);
    if (c.k1 != c.n_emb + parts * c.ns) return DDP_E_SHAPE;
    if ((e.p1 && !e.i1) || (e.p2 && !e.i2)) return DDP_E_ARG;
    if (c.n_groups <= 0 || c.n_groups > 64) return DDP_E_SHAPE;
    if (e.edge_cap <= 0) return 0;
    const int ctab_len = c.ctab_len;
    if (ctab_len <= 0 || ctab_len > 64 * 125) return DDP_E_SHAPE;
    const bool small = e.edge_cap <= 8 * 2 * ddp_num_sms();          // few edges: 8-edge tiles keep all SMs busy
    const int TE = small ? 8 : 32;
    const size_t smem = ((size_t)(c.k1 + c.hid + c.f_in + c.sh_dim + c.f_out * (FIXED ? 2 : 1)) * (TE + 4) + ctab_len) * sizeof(float) + TE * sizeof(int);
    if (smem > 200 * 1024) return DDP_E_SHAPE;
    static size_t configured[DDP_MAX_DEVICES][2] = {{0, 0}};      // largest opt-in so far, per device and tile size (per FIXED)
    size_t &cfg = configured[ddp_current_device()][small];
    if (smem > cfg) {
        cudaError_t err = small ? cudaFuncSetAttribute(tpconv_fp32_kernel<8, FIXED>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                                : cudaFuncSetAttribute(tpconv_fp32_kernel<32, FIXED>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (err != cudaSuccess) return (int)err;
        cfg = smem;
    }
    int tiles = (e.edge_cap + TE - 1) / TE;
    int grid = tiles < 2 * ddp_num_sms() ? tiles : 2 * ddp_num_sms();
    if (small) tpconv_fp32_kernel<8, FIXED><<<grid, NT, smem, (cudaStream_t)stream>>>(c, e, ctab_len, sum, status);
    else tpconv_fp32_kernel<32, FIXED><<<grid, NT, smem, (cudaStream_t)stream>>>(c, e, ctab_len, sum, status);
    DDP_LAUNCH_CHECK();
    return 0;
}

extern "C" int ddp_tpconv_fp32(const ddp_tpconv_t *conv, const ddp_tpconv_edges_t *edges, float *sum, void *stream) {
    return tpconv_fp32<false>(conv, edges, sum, nullptr, stream);
}

extern "C" int ddp_tpconv_fp32_fixed(const ddp_tpconv_t *conv, const ddp_tpconv_edges_t *edges, int64_t *sum, uint32_t *status,
                                     void *stream) {
    return tpconv_fp32<true>(conv, edges, reinterpret_cast<float *>(sum), status, stream);
}
