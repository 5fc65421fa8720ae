// Backward of the tensor product of a TensorProductConvLayer (training path, SURVEY 8(f) row 3): the gradient of
//   out_e[o][k] = sum_{u,i,j} w_e[u][o] C[i][j][k] x_{gather(e)}[u][i] sh_e[j]          (models/layers.py:40-85, e3nn FCTP)
// with respect to the per-edge weights w_e, the gathered node features x and the edge harmonics sh, for every row
// group of the conv's table-driven spec (the same ddp_tp_group_t / coefficient table the forward kernels use).
// The edge MLP around it (two Linears, ReLU) and the weight-gradient GEMMs  g_W2 = g_w^T h,  g_h = g_w W2  are plain
// library GEMMs on the host-mirror side (diffdock_pocket_b200/score_model.py:_ConvFn); this kernel is the part no
// library has.  Unlike the forward, the per-edge weights and their gradients ARE materialised here, in chunks of edges
// ([chunk][w_numel] fp32, like the reference's autograd does for the whole batch): a first correct backward, HBM-bound
// (2 x 4 B x w_numel per edge), not the fused tensor-core form of the forward.
//
// One thread per (edge, input row u of a group): it walks the group's mul_out weight columns of that row, so the
// contributions to g_x[u] / g_sh are summed in registers and leave with d1 + d2 atomics per thread.  FIXED
// (ddp_tp_backward_fixed): those atomics add int64 fixed point (DDP_ACC_FIXED_SHIFT), so the gradients do not depend on
// the order in which the threads of one node / edge arrive.
#include "ddp_common.cuh"

namespace {

constexpr int kMaxGroups = 64;
constexpr int kMaxD = 5;      // 2l + 1 for l <= 2

template <bool FIXED>
__global__ void __launch_bounds__(256)
tp_bwd_kernel(const ddp_tp_group_t *__restrict__ groups, int n_groups, const float *__restrict__ ctab, int rows_per_edge,
              const float *__restrict__ x, const int32_t *__restrict__ gather, int ldx,
              const float *__restrict__ sh, int sh_dim, const float *__restrict__ w, int w_numel,
              const float *__restrict__ g_out, int f_out, int n_edges,
              float *__restrict__ g_w, float *__restrict__ g_x, float *__restrict__ g_sh, uint32_t *status) {
    __shared__ ddp_tp_group_t sg[kMaxGroups];
    __shared__ int row_start[kMaxGroups + 1];
    if (threadIdx.x < n_groups) sg[threadIdx.x] = groups[threadIdx.x];
    __syncthreads();
    if (threadIdx.x == 0) {
        int acc = 0;
        for (int g = 0; g < n_groups; ++g) { row_start[g] = acc; acc += sg[g].mul_in; }
        row_start[n_groups] = acc;
    }
    __syncthreads();
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (tid >= (long long)n_edges * rows_per_edge) return;
    const int e = (int)(tid / rows_per_edge), row = (int)(tid % rows_per_edge);
    int gi = 0;
    while (gi + 1 < n_groups && row >= row_start[gi + 1]) ++gi;
    const ddp_tp_group_t g = sg[gi];
    const int u = row - row_start[gi];
    if (g.d1 > kMaxD || g.d2 > kMaxD || g.d_out > kMaxD) return;      // outside the contract (l <= 2): leave the gradients untouched
    const float *cg = ctab + g.c_off;
    const int node = gather[e];
    float xv[kMaxD], sv[kMaxD];
    for (int i = 0; i < g.d1; ++i) xv[i] = x[(size_t)node * ldx + g.x_off + u * g.d1 + i];
    for (int j = 0; j < g.d2; ++j) sv[j] = sh[(size_t)e * sh_dim + g.sh_off + j];
    // b[k] = sum_ij C x_i s_j (the forward basis);  T[i][k] = sum_j C s_j;  S[j][k] = sum_i C x_i
    float b[kMaxD], T[kMaxD][kMaxD], S[kMaxD][kMaxD];
    for (int k = 0; k < g.d_out; ++k) {
        b[k] = 0.f;
        for (int i = 0; i < g.d1; ++i) T[i][k] = 0.f;
        for (int j = 0; j < g.d2; ++j) S[j][k] = 0.f;
    }
    for (int i = 0; i < g.d1; ++i)
        for (int j = 0; j < g.d2; ++j)
            for (int k = 0; k < g.d_out; ++k) {
                const float c = cg[(i * g.d2 + j) * g.d_out + k];
                b[k] = fmaf(c * xv[i], sv[j], b[k]);
                T[i][k] = fmaf(c, sv[j], T[i][k]);
                S[j][k] = fmaf(c, xv[i], S[j][k]);
            }
    float gx[kMaxD], gs[kMaxD];
    for (int i = 0; i < kMaxD; ++i) { gx[i] = 0.f; gs[i] = 0.f; }
    const float *wr = w + (size_t)e * w_numel + g.w_off + (size_t)u * g.mul_out;
    float *gwr = g_w + (size_t)e * w_numel + g.w_off + (size_t)u * g.mul_out;
    const float *go = g_out + (size_t)e * f_out + g.out_off;
    for (int o = 0; o < g.mul_out; ++o) {
        const float wv = wr[o];
        float acc = 0.f;
        for (int k = 0; k < g.d_out; ++k) {
            const float gk = go[o * g.d_out + k];
            acc = fmaf(b[k], gk, acc);
            const float t = wv * gk;
            for (int i = 0; i < g.d1; ++i) gx[i] = fmaf(T[i][k], t, gx[i]);
            for (int j = 0; j < g.d2; ++j) gs[j] = fmaf(S[j][k], t, gs[j]);
        }
        gwr[o] = acc;
    }
    if (FIXED) {
        unsigned long long *qx = reinterpret_cast<unsigned long long *>(g_x), *qs = reinterpret_cast<unsigned long long *>(g_sh);
        if (qx != nullptr)
            for (int i = 0; i < g.d1; ++i) atomicAdd(qx + (size_t)node * ldx + g.x_off + u * g.d1 + i, ddp_to_fixed(gx[i], status));
        if (qs != nullptr)
            for (int j = 0; j < g.d2; ++j) atomicAdd(qs + (size_t)e * sh_dim + g.sh_off + j, ddp_to_fixed(gs[j], status));
        return;
    }
    if (g_x != nullptr)
        for (int i = 0; i < g.d1; ++i) atomicAdd(g_x + (size_t)node * ldx + g.x_off + u * g.d1 + i, gx[i]);
    if (g_sh != nullptr)
        for (int j = 0; j < g.d2; ++j) atomicAdd(g_sh + (size_t)e * sh_dim + g.sh_off + j, gs[j]);
}

__global__ void fixed_to_float_kernel(const long long *__restrict__ src, long long n, float *__restrict__ dst) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        dst[i] = ddp_from_fixed(src[i]);
}

}  // namespace

template <bool FIXED>
static int tp_backward(const ddp_tpconv_t *conv, int32_t rows_per_edge, const float *x, const int32_t *gather, int32_t ldx,
                       const float *sh, const float *w, const float *g_out, int32_t n_edges, float *g_w, float *g_x, float *g_sh,
                       uint32_t *status, void *stream) {
    if (!conv || !x || !gather || !sh || !w || !g_out || !g_w || (FIXED && !status)) return DDP_E_ARG;
    const ddp_tpconv_t &c = *conv;
    if (!c.groups || !c.ctab) return DDP_E_ARG;
    if (c.n_groups <= 0 || c.n_groups > kMaxGroups || rows_per_edge <= 0) return DDP_E_SHAPE;
    if (n_edges <= 0) return 0;
    // rows_per_edge = sum of mul_in over the groups (the groups themselves live on the device; irrep dimensions <= 5, i.e.
    // l <= 2, are the caller's contract -- the host mirror checks them against its spec)
    const long long total = (long long)n_edges * rows_per_edge;
    const int grid = (int)((total + 255) / 256);
    tp_bwd_kernel<FIXED><<<grid, 256, 0, (cudaStream_t)stream>>>(c.groups, c.n_groups, c.ctab, rows_per_edge, x, gather, ldx, sh, c.sh_dim,
                                                                 w, c.w_numel, g_out, c.f_out, n_edges, g_w, g_x, g_sh, status);
    DDP_LAUNCH_CHECK();
    return 0;
}

extern "C" int ddp_tp_backward(const ddp_tpconv_t *conv, int32_t rows_per_edge, const float *x, const int32_t *gather, int32_t ldx,
                               const float *sh, const float *w, const float *g_out, int32_t n_edges, float *g_w, float *g_x, float *g_sh,
                               void *stream) {
    return tp_backward<false>(conv, rows_per_edge, x, gather, ldx, sh, w, g_out, n_edges, g_w, g_x, g_sh, nullptr, stream);
}

extern "C" int ddp_tp_backward_fixed(const ddp_tpconv_t *conv, int32_t rows_per_edge, const float *x, const int32_t *gather, int32_t ldx,
                                     const float *sh, const float *w, const float *g_out, int32_t n_edges, float *g_w, int64_t *g_x,
                                     int64_t *g_sh, uint32_t *status, void *stream) {
    return tp_backward<true>(conv, rows_per_edge, x, gather, ldx, sh, w, g_out, n_edges, g_w, reinterpret_cast<float *>(g_x),
                             reinterpret_cast<float *>(g_sh), status, stream);
}

extern "C" int ddp_fixed_to_float(const int64_t *src, int64_t n, float *dst, void *stream) {
    if (!src || !dst || n < 0) return DDP_E_ARG;
    if (n == 0) return 0;
    const long long blocks = (n + 255) / 256;
    const int grid = (int)(blocks < 8 * ddp_num_sms() ? blocks : 8 * ddp_num_sms());
    fixed_to_float_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const long long *>(src), (long long)n, dst);
    DDP_LAUNCH_CHECK();
    return 0;
}
