// Pose checks of docked poses (DESIGN section 11): symmetry-corrected RMSD against a reference and steric-clash
// screening.  Both kernels are reductions whose results do not depend on the launch shape: the RMSD kernel reduces each
// pose inside one CTA in a fixed order, the clash kernel adds integers and takes minima (atomicMin on the bits of
// non-negative floats), so every output is bitwise reproducible and independent of how poses are packed into launches.
#include "ddp_common.cuh"

namespace {

constexpr int kMaxRows = 512;                  // = ddp_pose_max_ligand_atoms(): pose and reference rows live in shared memory
constexpr int kRmsdThreads = 256;
constexpr int kRmsdWarps = kRmsdThreads / 32;
constexpr int kClashThreads = 128;             // pocket (or ligand) atoms per CTA: one per thread
// A pair is looked at closely only if it clashes or may lower the thread's minimum ratio.  The cheap test compares d^2
// with (best * s)^2, whose three roundings are far below this slack, so no pair that lowers the minimum is skipped.
constexpr float kFilterSlack = 1.00001f;

__global__ void __launch_bounds__(kRmsdThreads)
pose_rmsd_kernel(const float *__restrict__ pos, const int32_t *__restrict__ pos_ptr, const int32_t *__restrict__ pose_complex,
                 const float *__restrict__ ref, const int32_t *__restrict__ ref_off, const int16_t *__restrict__ autos,
                 const int32_t *__restrict__ auto_off, const int32_t *__restrict__ n_auto, float *__restrict__ rmsd,
                 int32_t *__restrict__ best) {
    __shared__ float s_x[3 * kMaxRows], s_r[3 * kMaxRows];
    __shared__ double s_msd[kRmsdWarps];
    __shared__ int s_a[kRmsdWarps];
    const int p = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int c = pose_complex[p];
    const int r0 = pos_ptr[p], n = pos_ptr[p + 1] - r0;
    if (n <= 0 || n > kMaxRows) {              // the host checks the cap; a row it let through reads as NaN, never as a value
        if (tid == 0) { rmsd[p] = n == 0 ? 0.f : __int_as_float(0x7fc00000); best[p] = n == 0 ? 0 : -1; }
        return;
    }
    const float *x = pos + 3 * (size_t)r0, *r = ref + 3 * (size_t)ref_off[c];
    for (int k = tid; k < 3 * n; k += kRmsdThreads) { s_x[k] = x[k]; s_r[k] = r[k]; }
    __syncthreads();
    const int na = n_auto[c];
    const int16_t *tab = autos + auto_off[c];
    double bmsd = INFINITY;
    int ba = 0x7fffffff;
    for (int a = warp; a < na; a += kRmsdWarps) {   // warp w: automorphisms w, w + 8, ... (ascending: the first minimum wins)
        const int16_t *perm = tab + (size_t)a * n;
        double acc = 0.0;
        for (int i = lane; i < n; i += 32) {
            const int j = perm[i];
            const double dx = (double)s_x[3 * i] - (double)s_r[3 * j];
            const double dy = (double)s_x[3 * i + 1] - (double)s_r[3 * j + 1];
            const double dz = (double)s_x[3 * i + 2] - (double)s_r[3 * j + 2];
            acc += dx * dx + dy * dy + dz * dz;
        }
        for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);   // same bits in every lane
        if (acc < bmsd) { bmsd = acc; ba = a; }
    }
    if (lane == 0) { s_msd[warp] = bmsd; s_a[warp] = ba; }
    __syncthreads();
    if (tid == 0) {
        double m = s_msd[0];
        int am = s_a[0];
        for (int w = 1; w < kRmsdWarps; ++w)
            if (s_msd[w] < m || (s_msd[w] == m && s_a[w] < am)) { m = s_msd[w]; am = s_a[w]; }
        rmsd[p] = (float)sqrt(m / n);
        best[p] = am;
    }
}

// One pair of a clash set: count it if d^2 < (ratio s)^2 and keep the minimum of d / s, s = R_i + R_j.  `keep` decides,
// only for the pairs that pass the cheap test, whether the pair belongs to the set.
template <typename Keep>
__device__ __forceinline__ void clash_pair(float ax, float ay, float az, float ar, float4 b, float ratio, int &cnt, float &best,
                                           Keep keep) {
    const float dx = __fsub_rn(ax, b.x), dy = __fsub_rn(ay, b.y), dz = __fsub_rn(az, b.z);
    const float d2 = __fmaf_rn(dz, dz, __fmaf_rn(dy, dy, __fmul_rn(dx, dx)));
    const float s = __fadd_rn(ar, b.w), t = __fmul_rn(ratio, s), u = __fmul_rn(best, s);
    const bool clash = d2 < __fmul_rn(t, t);
    if ((clash || d2 < __fmul_rn(__fmul_rn(u, u), kFilterSlack)) && keep()) {
        cnt += clash;
        best = fminf(best, __fdiv_rn(__fsqrt_rn(d2), s));
    }
}

__device__ __forceinline__ void clash_flush(int cnt, float best, int32_t *count, float *min_ratio) {
    for (int o = 16; o; o >>= 1) {
        cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
        best = fminf(best, __shfl_xor_sync(0xffffffffu, best, o));
    }
    if ((threadIdx.x & 31) == 0) {
        if (cnt) atomicAdd(count, cnt);
        if (best < INFINITY) atomicMin(reinterpret_cast<unsigned int *>(min_ratio), __float_as_uint(best));
    }
}

// grid (n_poses, chunks): chunk y < ceil(N_a / 128) takes pocket atoms [128 y, 128 y + 128) against the ligand and the moved
// side-chain atoms; the next ceil(N_l / 128) chunks take ligand atoms against the ligand atoms after them.
__global__ void __launch_bounds__(kClashThreads) clash_kernel(ddp_clash_screen_t A) {
    __shared__ float4 s_l[kMaxRows];
    __shared__ float4 s_m[kClashThreads];
    __shared__ int s_mo[kClashThreads];
    const int p = blockIdx.x, chunk = blockIdx.y, tid = threadIdx.x;
    const ddp_clash_complex_t C = A.complexes[A.pose_complex[p]];
    const int l0 = A.lig_ptr[p], nl = A.lig_ptr[p + 1] - l0;
    const int a0 = A.atom_ptr[p], na = A.atom_ptr[p + 1] - a0;
    const int n_pc = (na + kClashThreads - 1) / kClashThreads, n_lc = (nl + kClashThreads - 1) / kClashThreads;
    if (chunk >= n_pc + n_lc) return;
    if (nl > kMaxRows) {                       // the host checks the cap; a row it let through reads as count -1
        if (chunk == 0 && tid < 3) A.count[3 * p + tid] = -1;
        return;
    }
    for (int i = tid; i < nl; i += kClashThreads) {
        const float *q = A.lig_pos + 3 * (size_t)(l0 + i);
        s_l[i] = make_float4(q[0], q[1], q[2], A.radius[A.lig_type[C.lig_type_off + i]]);
    }
    __syncthreads();
    const float ratio = A.ratio;
    if (chunk < n_pc) {
        const int j = chunk * kClashThreads + tid;
        const bool act = j < na;
        float px = 0.f, py = 0.f, pz = 0.f, pr = 0.f;
        int own = -1;
        if (act) {
            const float *q = A.atom_pos + 3 * (size_t)(a0 + j);
            px = q[0]; py = q[1]; pz = q[2];
            pr = A.radius[A.atom_type[C.atom_off + j]];
            own = A.atom_owner[C.atom_off + j];
        }
        int cnt = 0;
        float best = INFINITY;
        if (act)
            for (int i = 0; i < nl; ++i) clash_pair(px, py, pz, pr, s_l[i], ratio, cnt, best, [] { return true; });
        clash_flush(cnt, best, A.count + 3 * p, A.min_ratio + 3 * p);
        cnt = 0;
        best = INFINITY;
        for (int m0 = 0; m0 < C.n_moved; m0 += kClashThreads) {
            const int nt = min(kClashThreads, C.n_moved - m0);
            __syncthreads();
            if (tid < nt) {
                const int k = A.moved[C.moved_off + m0 + tid];
                const float *q = A.atom_pos + 3 * (size_t)(a0 + k);
                s_m[tid] = make_float4(q[0], q[1], q[2], A.radius[A.atom_type[C.atom_off + k]]);
                s_mo[tid] = A.atom_owner[C.atom_off + k];
            }
            __syncthreads();
            if (act)
                for (int t = 0; t < nt; ++t)
                    clash_pair(px, py, pz, pr, s_m[t], ratio, cnt, best, [&] {
                        if (s_mo[t] == own) return false;
                        const int32_t *e = A.excl + 2 * (size_t)C.excl_off;
                        for (int k = 0; k < C.n_excl; ++k)
                            if (e[2 * k] == m0 + t && e[2 * k + 1] == j) return false;
                        return true;
                    });
        }
        clash_flush(cnt, best, A.count + 3 * p + 1, A.min_ratio + 3 * p + 1);
    } else {
        const int i = (chunk - n_pc) * kClashThreads + tid;
        int cnt = 0;
        float best = INFINITY;
        if (i < nl) {
            const float4 me = s_l[i];
            const uint32_t *row = A.far_mask + C.far_off + (size_t)i * ((nl + 31) >> 5);
            for (int j = i + 1; j < nl; ++j)
                clash_pair(me.x, me.y, me.z, me.w, s_l[j], ratio, cnt, best, [&] { return ((row[j >> 5] >> (j & 31)) & 1u) != 0; });
        }
        clash_flush(cnt, best, A.count + 3 * p + 2, A.min_ratio + 3 * p + 2);
    }
}

}  // namespace

extern "C" int ddp_pose_rmsd(const float *pos, const int32_t *pos_ptr, const int32_t *pose_complex, int32_t n_poses,
                             const float *ref, const int32_t *ref_off, const int16_t *autos, const int32_t *auto_off,
                             const int32_t *n_auto, float *rmsd, int32_t *best, void *stream) {
    if (n_poses < 0) return DDP_E_SHAPE;
    if (n_poses == 0) return 0;
    if (!pos || !pos_ptr || !pose_complex || !ref || !ref_off || !autos || !auto_off || !n_auto || !rmsd || !best) return DDP_E_ARG;
    pose_rmsd_kernel<<<n_poses, kRmsdThreads, 0, (cudaStream_t)stream>>>(pos, pos_ptr, pose_complex, ref, ref_off, autos, auto_off,
                                                                         n_auto, rmsd, best);
    DDP_LAUNCH_CHECK();
    return 0;
}

extern "C" int ddp_clash_screen(const ddp_clash_screen_t *args, void *stream) {
    if (!args) return DDP_E_ARG;
    const ddp_clash_screen_t &A = *args;
    if (A.n_poses < 0 || A.max_lig_atoms < 0 || A.max_atoms < 0 || !(A.ratio >= 0.f)) return DDP_E_SHAPE;
    if (A.n_poses == 0) return 0;
    if (!A.pose_complex || !A.lig_pos || !A.lig_ptr || !A.atom_pos || !A.atom_ptr || !A.complexes || !A.lig_type ||
        !A.atom_type || !A.atom_owner || !A.far_mask || !A.radius || !A.count || !A.min_ratio)
        return DDP_E_ARG;
    const int chunks = (A.max_atoms + kClashThreads - 1) / kClashThreads + (A.max_lig_atoms + kClashThreads - 1) / kClashThreads;
    if (chunks == 0) return 0;
    if (chunks > 65535) return DDP_E_SHAPE;
    clash_kernel<<<dim3(A.n_poses, chunks), kClashThreads, 0, (cudaStream_t)stream>>>(A);
    DDP_LAUNCH_CHECK();
    return 0;
}
