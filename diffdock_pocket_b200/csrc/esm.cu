// ESM-2 receptor embeddings (DESIGN section 12): the element-wise stages around the library GEMMs and a fused rotary
// multi-head attention.  Every output element is written by one thread in a fixed order (warp-shuffle trees, no atomics
// on floating-point data), so results are bitwise repeatable and do not depend on how many sequences share a launch.
#include "ddp_common.cuh"

namespace {

constexpr int kHd = 64;                 // head dimension (ESM-2 650M: 1280 / 20)
constexpr int kHalf = kHd / 2;          // rotary frequencies
constexpr int kMaxT = 1024;             // 1022 residues + BOS + EOS
constexpr int kBq = 64, kBk = 64;       // query rows per CTA, keys per tile
constexpr int kAttThreads = 256;        // 16 x 16 threads, each a 4 x 4 block of the score and output tiles
constexpr int kLd = kHd + 4;            // shared row stride (floats): float4-aligned, staggers the transposed stores
constexpr size_t kAttSmem = 4 * kHd * kLd * sizeof(float);
constexpr int kRowThreads = 256;        // layer norm / embedding: one warp per row
constexpr int kLnMaxVec = 16;           // float4 per lane: layer-norm rows of up to 32 * 4 * 16 = 2048 columns
// fair-esm ESM2.forward: x * (1 - 0.15 * 0.8) / (1 - mask_ratio_observed), the Python factor rounded to fp32 as torch does
constexpr float kKeep = (float)(1.0 - 0.15 * 0.8);

struct RotaryTable { float inv_freq[kHalf]; };

__device__ __forceinline__ float warp_sum(float v) {
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// fair-esm ESM2.forward (esm/model/esm2.py): embed_tokens, token-dropout rescaling, <mask> and pad rows zeroed.
// grid (ceil(T / 8), B): every CTA counts its sequence's tokens itself (integer counts, no cross-CTA traffic).
__global__ void __launch_bounds__(kRowThreads)
esm_embed_kernel(const int64_t *__restrict__ tokens, int T, const float *__restrict__ weight, int vocab, int D, int pad_idx,
                 int mask_idx, float *__restrict__ out) {
    __shared__ int s_cnt[2];
    const int b = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t *tok = tokens + (size_t)b * T;
    if (tid < 2) s_cnt[tid] = 0;
    __syncthreads();
    int n_mask = 0, n_valid = 0;
    for (int t = tid; t < T; t += kRowThreads) {
        const int64_t v = tok[t];
        n_mask += v == mask_idx;
        n_valid += v != pad_idx;
    }
    for (int o = 16; o; o >>= 1) {
        n_mask += __shfl_xor_sync(0xffffffffu, n_mask, o);
        n_valid += __shfl_xor_sync(0xffffffffu, n_valid, o);
    }
    if (lane == 0) { atomicAdd(&s_cnt[0], n_mask); atomicAdd(&s_cnt[1], n_valid); }
    __syncthreads();
    const float ratio = __fdiv_rn((float)s_cnt[0], (float)s_cnt[1]);
    const float denom = __fsub_rn(1.f, ratio);
    const int t = blockIdx.x * (kRowThreads / 32) + warp;
    if (t >= T) return;
    const int64_t v = tok[t];
    float *o = out + ((size_t)b * T + t) * D;
    if (v == pad_idx || v == mask_idx) {
        for (int c = lane; c < D; c += 32) o[c] = 0.f;
    } else if (v < 0 || v >= vocab) {        // the host validates tokens; a bad one reads as NaN, never as another row
        for (int c = lane; c < D; c += 32) o[c] = __int_as_float(0x7fc00000);
    } else {
        const float *w = weight + (size_t)v * D;
        for (int c = lane; c < D; c += 32) o[c] = __fdiv_rn(__fmul_rn(w[c], kKeep), denom);
    }
}

// One warp per row; the row stays in registers between the two statistics passes, so y may alias x.
__global__ void __launch_bounds__(kRowThreads)
layer_norm_kernel(float *__restrict__ x, const float *__restrict__ residual_bias, const float *__restrict__ gamma,
                  const float *__restrict__ beta, int rows, int cols, float eps, float *y) {
    const int row = blockIdx.x * (kRowThreads / 32) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= rows) return;
    float *xr = x + (size_t)row * cols;
    float4 v[kLnMaxVec];
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < kLnMaxVec; ++k) {
        const int c = (k * 32 + lane) * 4;
        if (c < cols) {
            v[k] = *reinterpret_cast<const float4 *>(xr + c);
            if (residual_bias) {
                const float4 r = *reinterpret_cast<const float4 *>(residual_bias + c);
                v[k].x += r.x; v[k].y += r.y; v[k].z += r.z; v[k].w += r.w;
                *reinterpret_cast<float4 *>(xr + c) = v[k];
            }
            s += (v[k].x + v[k].y) + (v[k].z + v[k].w);
        }
    }
    const float mean = warp_sum(s) / (float)cols;
    float q = 0.f;
#pragma unroll
    for (int k = 0; k < kLnMaxVec; ++k) {
        const int c = (k * 32 + lane) * 4;
        if (c < cols) {
            const float a = v[k].x - mean, b = v[k].y - mean, d = v[k].z - mean, e = v[k].w - mean;
            q += (a * a + b * b) + (d * d + e * e);
        }
    }
    const float rstd = rsqrtf(warp_sum(q) / (float)cols + eps);
    float *yr = y + (size_t)row * cols;
#pragma unroll
    for (int k = 0; k < kLnMaxVec; ++k) {
        const int c = (k * 32 + lane) * 4;
        if (c < cols) {
            const float4 g = *reinterpret_cast<const float4 *>(gamma + c), bb = *reinterpret_cast<const float4 *>(beta + c);
            float4 r;
            r.x = (v[k].x - mean) * rstd * g.x + bb.x;
            r.y = (v[k].y - mean) * rstd * g.y + bb.y;
            r.z = (v[k].z - mean) * rstd * g.z + bb.z;
            r.w = (v[k].w - mean) * rstd * g.w + bb.w;
            *reinterpret_cast<float4 *>(yr + c) = r;
        }
    }
}

__device__ __forceinline__ float gelu_erf(float v) { return 0.5f * v * (1.f + erff(v * 0.70710678118654752f)); }

__global__ void bias_gelu_kernel(float4 *__restrict__ x, const float4 *__restrict__ bias, int64_t n4, int cols4) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
        float4 v = x[i];
        const float4 b = bias[i % cols4];
        v.x = gelu_erf(v.x + b.x); v.y = gelu_erf(v.y + b.y); v.z = gelu_erf(v.z + b.z); v.w = gelu_erf(v.w + b.w);
        x[i] = v;
    }
}

// RotaryEmbedding (esm/rotary_embedding.py) of the pair (x[i], x[i + 32]) at position t: the angle float(t) * inv_freq[i]
// rounded once in fp32, then x * cos + rotate_half(x) * sin with its products and sum rounded separately, as torch does.
__device__ __forceinline__ void rope(float x1, float x2, int t, float f, float &o1, float &o2) {
    float s, c;
    sincosf(__fmul_rn((float)t, f), &s, &c);
    o1 = __fadd_rn(__fmul_rn(x1, c), __fmul_rn(-x2, s));
    o2 = __fadd_rn(__fmul_rn(x2, c), __fmul_rn(x1, s));
}

// Positions [r0, r0 + 64) of one head of the sequence starting at row0, rotated, stored transposed (sh[d][t - r0]);
// positions at or past `end` are zero.
// Thread `tid` always handles frequency i = tid % 32 (the stride is a multiple of 32): `freq` is inv_freq[i].
__device__ __forceinline__ void load_rotated(float *__restrict__ sh, const float *__restrict__ src, size_t row0, int ld, int r0,
                                             int end, float freq) {
    for (int e = threadIdx.x; e < 64 * kHalf; e += kAttThreads) {
        const int r = e >> 5, i = e & 31, t = r0 + r;
        float a = 0.f, c = 0.f;
        if (t < end) {
            const float *p = src + (row0 + t) * (size_t)ld;
            rope(__ldg(p + i), __ldg(p + i + kHalf), t, freq, a, c);
        }
        sh[i * kLd + r] = a;
        sh[(i + kHalf) * kLd + r] = c;
    }
}

// MultiheadAttention.forward with rotary embeddings and a key padding mask (esm/multihead_attention.py), one CTA per
// (64-query tile, head, sequence).  Online softmax over 64-key tiles: running row maxima m, sums l and the output tile
// O stay in registers, the scores of one tile pass through shared memory once as probabilities, and the [T, T] matrix
// is never written.  Score tile S = Q K^T and O += P V are 4 x 4 register blocks per thread over float4 shared reads.
__global__ void __launch_bounds__(kAttThreads, 2)
esm_attention_kernel(const float *__restrict__ q, const float *__restrict__ k, const float *__restrict__ v, int ld_in,
                     const int32_t *__restrict__ lengths, const __grid_constant__ RotaryTable rt, int T, float *__restrict__ out, int ld_out) {
    extern __shared__ float4 smem4[];
    float *sQ = reinterpret_cast<float *>(smem4);   // [d][query row]
    float *sK = sQ + kHd * kLd;                      // [d][key]
    float *sV = sK + kHd * kLd;                      // [key][d]
    float *sP = sV + kBk * kLd;                      // [key][query row]
    const int q0 = blockIdx.x * kBq, h = blockIdx.y, b = blockIdx.z, tid = threadIdx.x;
    const int tx = tid & 15, ty = tid >> 4;          // 16 threads of a half-warp share query rows ty * 4 .. + 3
    const int len = min(lengths[b], T);
    const size_t row0 = (size_t)b * T;
    const int hoff = h * kHd;
    const float freq = rt.inv_freq[tid & 31];       // read in place from the parameter bank (__grid_constant__: no local copy)
    load_rotated(sQ, q + hoff, row0, ld_in, q0, T, freq);
    float o[4][4], m[4], l[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        m[i] = -INFINITY; l[i] = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) o[i][j] = 0.f;
    }
    for (int k0 = 0; k0 < len; k0 += kBk) {
        __syncthreads();                             // the previous tile's sK / sV / sP reads are done (and sQ is written)
        load_rotated(sK, k + hoff, row0, ld_in, k0, len, freq);
        for (int e = tid; e < kBk * (kHd / 4); e += kAttThreads) {
            const int c = e >> 4, d4 = (e & 15) * 4;
            float4 val = make_float4(0.f, 0.f, 0.f, 0.f);
            if (k0 + c < len) val = __ldg(reinterpret_cast<const float4 *>(v + (row0 + k0 + c) * (size_t)ld_in + hoff + d4));
            *reinterpret_cast<float4 *>(sV + c * kLd + d4) = val;
        }
        __syncthreads();
        float s[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) s[i][j] = 0.f;
#pragma unroll 16
        for (int d = 0; d < kHd; ++d) {
            const float4 a = *reinterpret_cast<const float4 *>(sQ + d * kLd + ty * 4);
            const float4 bb = *reinterpret_cast<const float4 *>(sK + d * kLd + tx * 4);
            const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {bb.x, bb.y, bb.z, bb.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) s[i][j] = fmaf(av[i], bv[j], s[i][j]);
        }
        float p[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (k0 + tx * 4 + j >= len) s[i][j] = -INFINITY;     // key padding mask
            float mx = fmaxf(fmaxf(s[i][0], s[i][1]), fmaxf(s[i][2], s[i][3]));
            for (int o2 = 8; o2; o2 >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o2));
            const float mn = fmaxf(m[i], mx);                        // finite: key k0 < len is in every visited tile
            const float alpha = expf(m[i] - mn);
            float rs = 0.f;
#pragma unroll
            for (int j = 0; j < 4; ++j) { p[i][j] = expf(s[i][j] - mn); rs += p[i][j]; }
            for (int o2 = 8; o2; o2 >>= 1) rs += __shfl_xor_sync(0xffffffffu, rs, o2);
            l[i] = l[i] * alpha + rs;
            m[i] = mn;
#pragma unroll
            for (int j = 0; j < 4; ++j) o[i][j] *= alpha;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j)
            *reinterpret_cast<float4 *>(sP + (tx * 4 + j) * kLd + ty * 4) = make_float4(p[0][j], p[1][j], p[2][j], p[3][j]);
        __syncthreads();
#pragma unroll 16
        for (int c = 0; c < kBk; ++c) {
            const float4 a = *reinterpret_cast<const float4 *>(sP + c * kLd + ty * 4);
            const float4 bb = *reinterpret_cast<const float4 *>(sV + c * kLd + tx * 4);
            const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {bb.x, bb.y, bb.z, bb.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) o[i][j] = fmaf(av[i], bv[j], o[i][j]);
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int t = q0 + ty * 4 + i;
        if (t >= T) continue;
        const float inv = l[i] > 0.f ? 1.f / l[i] : 0.f;
        *reinterpret_cast<float4 *>(out + (row0 + t) * (size_t)ld_out + hoff + tx * 4) =
            make_float4(o[i][0] * inv, o[i][1] * inv, o[i][2] * inv, o[i][3] * inv);
    }
}

bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

}  // namespace

extern "C" int ddp_esm_embed(const int64_t *tokens, int32_t B, int32_t T, const float *weight, int32_t vocab, int32_t D,
                             int32_t pad_idx, int32_t mask_idx, float *out, void *stream) {
    if (B < 0 || T < 0 || vocab <= 0 || D <= 0 || B > 65535) return DDP_E_SHAPE;
    if (B == 0 || T == 0) return 0;
    if (!tokens || !weight || !out) return DDP_E_ARG;
    const dim3 grid((T + kRowThreads / 32 - 1) / (kRowThreads / 32), B);
    esm_embed_kernel<<<grid, kRowThreads, 0, (cudaStream_t)stream>>>(tokens, T, weight, vocab, D, pad_idx, mask_idx, out);
    DDP_LAUNCH_CHECK();
    return 0;
}

extern "C" int ddp_layer_norm(float *x, const float *residual_bias, const float *gamma, const float *beta, int32_t rows,
                              int32_t cols, float eps, float *y, void *stream) {
    if (rows < 0 || cols <= 0 || cols % 4 || cols > 32 * 4 * kLnMaxVec || !(eps > 0.f)) return DDP_E_SHAPE;
    if (rows == 0) return 0;
    if (!x || !gamma || !beta || !y) return DDP_E_ARG;
    if (residual_bias && y == x) return DDP_E_ARG;   // the updated residual stream would be overwritten by its norm
    if (!aligned16(x) || !aligned16(gamma) || !aligned16(beta) || !aligned16(y) || (residual_bias && !aligned16(residual_bias)))
        return DDP_E_ARG;
    const int per = kRowThreads / 32;
    layer_norm_kernel<<<(rows + per - 1) / per, kRowThreads, 0, (cudaStream_t)stream>>>(x, residual_bias, gamma, beta, rows, cols,
                                                                                        eps, y);
    DDP_LAUNCH_CHECK();
    return 0;
}

extern "C" int ddp_bias_gelu(float *x, const float *bias, int32_t rows, int32_t cols, void *stream) {
    if (rows < 0 || cols <= 0 || cols % 4) return DDP_E_SHAPE;
    if (rows == 0) return 0;
    if (!x || !bias) return DDP_E_ARG;
    if (!aligned16(x) || !aligned16(bias)) return DDP_E_ARG;
    const int64_t n4 = (int64_t)rows * cols / 4;
    const int64_t cap = (int64_t)ddp_num_sms() * 8, want = (n4 + 255) / 256;
    const int blocks = (int)(want < cap ? want : cap);
    bias_gelu_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<float4 *>(x), reinterpret_cast<const float4 *>(bias),
                                                              n4, cols / 4);
    DDP_LAUNCH_CHECK();
    return 0;
}

extern "C" int ddp_esm_attention(const float *q, const float *k, const float *v, int32_t ld_in, const int32_t *lengths,
                                 const float *inv_freq_host, int32_t B, int32_t T, int32_t H, int32_t head_dim, float *out,
                                 int32_t ld_out, void *stream) {
    if (head_dim != kHd) return DDP_E_UNSUPPORTED;
    if (B < 0 || T < 0 || H < 0 || T > kMaxT || B > 65535 || H > 65535) return DDP_E_SHAPE;
    if (ld_in < H * kHd || ld_out < H * kHd || ld_in % 4 || ld_out % 4) return DDP_E_SHAPE;
    if (B == 0 || T == 0 || H == 0) return 0;
    if (!q || !k || !v || !lengths || !inv_freq_host || !out) return DDP_E_ARG;
    if (!aligned16(v) || !aligned16(out)) return DDP_E_ARG;
    static bool opted[DDP_MAX_DEVICES] = {false};
    cudaError_t e = ddp_smem_opt_in(esm_attention_kernel, kAttSmem, opted);
    if (e != cudaSuccess) return (int)e;
    RotaryTable rt;
    for (int i = 0; i < kHalf; ++i) rt.inv_freq[i] = inv_freq_host[i];
    const dim3 grid((T + kBq - 1) / kBq, H, B);
    esm_attention_kernel<<<grid, kAttThreads, kAttSmem, (cudaStream_t)stream>>>(q, k, v, ld_in, lengths, rt, T, out, ld_out);
    DDP_LAUNCH_CHECK();
    return 0;
}
