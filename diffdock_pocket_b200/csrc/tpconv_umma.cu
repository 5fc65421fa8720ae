// Tensor-core tensor-product convolution for sm_100a: tcgen05.mma (bf16 x bf16 -> fp32 in TMEM),
// weights streamed by TMA bulk copies (cp.async.bulk, UBLKCP) through an mbarrier ring, per-edge
// weight tiles consumed straight out of TMEM by the tensor-product epilogue.  The per-edge weight
// vector (up to 10000 floats) never exists in shared or global memory.
//
// One CTA (persistent, one per SM) walks 128-edge tiles (TMEM lane = edge) of up to 9 convolutions that share
// irreps (the convs of one interaction layer): tile g of the launch belongs to job j with pref[j] <= g < pref[j+1].
// Warp roles (384 threads = three warpgroups; setmaxnreg moves registers from the middle one to the two epilogue ones):
//   warps 0-3 and 8-11  epilogue, one warpgroup per TMEM accumulator (TMEM lane = edge in both): warpgroup g handles the
//              weight tiles that land in accumulator g, i.e. every other tile of the image's tile order, with its own
//              per-edge output registers.  Per weight tile: tcgen05.ld the [128 x N] accumulator, multiply with the
//              tensor-product basis (node features fetched from global memory into registers one own tile ahead) and
//              accumulate the edge's output in registers; when the warpgroup's next tile belongs to another output
//              block, a warp-level segmented pre-reduction over runs of equal aggregation nodes, then vector
//              red.global.add.  The packer interleaves the tiles of the first and the second half of the output blocks
//              so that each warpgroup normally owns whole blocks (no duplicated atomics).  Warpgroup 0 also turns the
//              GEMM1 result into the A operand of GEMM2 (ReLU, bf16, core-matrix order), after its last flush and the
//              next edge tile's per-edge set-up, which fit into the wait for that GEMM1.
//              Why two: the epilogue is a chain of dependent instructions (tile decode, basis, TMEM round trips) on ONE
//              warp per scheduler, ~1350 cycles per scalar tile and ~2500 per vector tile against 1440 / 1250 cycles of
//              MMAs (profiles/r2_umma_timeline_*.txt): a single warpgroup was busy 93 % of the time and set the pace.
//   warp 4     TMA producer: streams the pre-packed weight image (already in UMMA core-matrix order and in
//              consumption order) slab by slab.
//   warps 5, 7 MMA issuers (one elected lane each), one per TMEM accumulator, so that one of them is always parked on
//              the tensor pipe's queue while the other does its per-tile barrier work; warp 5 also allocates TMEM.
//   warp 6     gather: stage [emb | node scalars] of the NEXT edge tile as the bf16 A operand (double buffered),
//              so the gather latency hides under the current tile's GEMM2.
//
// Biases ride in the GEMMs: A has a constant-one column (padding slot of the first 64-wide source block)
// and the images carry b1 / b2 in that K row; the hidden unit `hid` regenerates the one for GEMM2.
// mode 1 ("bf16x3") splits both operands into bf16 hi + lo and issues hi*hi + lo*hi + hi*lo, which gives
// fp32-grade products (error ~2^-17 per product) for the 1e-4 parity gate.
#include <cuda_bf16.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "ddp_common.cuh"

namespace umma {

constexpr int TILE_M = 128;
constexpr uint32_t MAGIC = 0x44445055u;  // "DDPU"

struct TileDesc {
    uint16_t n_cols;      // UMMA N of this weight tile (multiple of 16): n_rows * mul_out rounded up, rest zero padding
    uint8_t kind;         // basis of every row of the tile: 0 x*s0, 1 dot(xv,s1), 2 x*s1, 3 xv*s0, 4 cross(xv,s1),
                          // 5 (sh_lmax = 2 only) C(1,2,1)(xv, s2): the l = 2 harmonics as a 3 x 3 matrix applied to xv
    uint8_t n_rows;       // basis rows covered
    uint16_t out_off;     // first output feature of the block
    uint8_t flags;        // bit 0: first tile of its block; bit 1: swap the last input irrep into slot 0 first; bit 2: last tile
    uint8_t ctab5;        // kind 5: which 45-float coupling table of the image (Header::ctab5_off)
    uint16_t x_off;       // slot of the first input feature of row 0 (row rr reads x_off + rr * (kind 0/2 ? 1 : 3))
    uint16_t pad1;
    uint32_t pad2;
};
static_assert(sizeof(TileDesc) == 16, "TileDesc is read as one 16-byte word");

struct Header {
    uint32_t magic;
    int32_t mode, ns, nv, ks, kp, n1, stage_k, n_tiles, n_slabs_per_edge_tile;
    int32_t f_in, f_out, n_parts;
    int32_t slab_elems_max;   // elements (bf16) of the largest slab part (one of hi / lo)
    int64_t tiles_off, slabs_off, total_bytes;
    int32_t sh_dim, n_ctab5;  // 4 (sh_lmax 1) or 9 (sh_lmax 2); coupling tables [i][j][k] (3 x 5 x 3 floats each) of the kind-5 groups
    int64_t ctab5_off;
};

__host__ __device__ inline int slab_bytes(int n_cols, int stage_k, int mode) { return n_cols * stage_k * 2 * (mode ? 2 : 1); }

// ------------------------------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "W_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@!p bra W_%=;\n\t}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// Waits with slack (the gather warp is a whole edge tile ahead, the TMA producer a ring of slabs): let the hardware park
// the warp (suspend-time hint) and back off between polls instead of spinning -- in profiles/r1_ncu_umma_v23_summary.txt
// the plain try_wait loops of these two roles are 22 % of all executed warp instructions, i.e. issue energy under a
// power cap.  The latency-critical waits (issuers, epilogue) use the hint without the back-off (-DDDP_UMMA_SPIN restores
// the plain loops).
template <int SLEEP_NS>
__device__ __forceinline__ void mbar_wait_relaxed(uint64_t *bar, uint32_t parity) {
    uint32_t done;
    for (;;) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}\n"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity), "r"(20000u)
            : "memory");
        if (done) break;
        if (SLEEP_NS > 0) __nanosleep(SLEEP_NS);
    }
}
// Debug build (-DDDP_UMMA_WATCHDOG, with -DDDP_UMMA_TRACE): a wait that has polled ~2^18 times records
// (code, a, b, barrier parity asked for) of its warp in the host-visible trace buffer, so a deadlock can be read
// from the host while the kernel still hangs (scripts/umma_watchdog.py).
#ifdef DDP_UMMA_WATCHDOG
__device__ __forceinline__ void mbar_wait_wd(uint64_t *bar, uint32_t parity, long long *trace, int code, int a, int b) {
    uint32_t done = 0;
    unsigned long long polls = 0;
    while (!done) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}\n"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
        if (!done && ++polls == (1ull << 18) && trace != nullptr && (threadIdx.x & 31) == 0) {
            long long *rec = trace + ((size_t)blockIdx.x * 12 + (threadIdx.x >> 5)) * 4;   // 12 warps per CTA
            rec[0] = code; rec[1] = a; rec[2] = b; rec[3] = parity;
            __threadfence_system();
        }
    }
}
#define DDP_WAIT(bar, par, code, a, b) mbar_wait_wd(bar, par, jobs.trace, code, a, b)
#else
#ifdef DDP_UMMA_SPIN
#define DDP_WAIT(bar, par, code, a, b) mbar_wait(bar, par)
#else
#define DDP_WAIT(bar, par, code, a, b) mbar_wait_relaxed<0>(bar, par)   // suspend-time hint, no back-off: wakes on completion
#endif
#endif
#if defined(DDP_UMMA_WATCHDOG) || defined(DDP_UMMA_SPIN)
#define DDP_WAIT_RELAXED(SLEEP, bar, par, code, a, b) DDP_WAIT(bar, par, code, a, b)
#else
#define DDP_WAIT_RELAXED(SLEEP, bar, par, code, a, b) mbar_wait_relaxed<SLEEP>(bar, par)
#endif
// Split-phase barrier test for the MMA issue loop: mbar_test_pN starts a non-blocking phase test whose predicate
// lives in a PTX register declared once per kernel (DDP_DECLARE_TEST_PREDS); mbar_finish_pN consumes it later (falling
// back to the blocking wait), so the ~100-cycle shared-memory round trip overlaps the tcgen05.mma issue in between.
#define DDP_DECLARE_TEST_PREDS() asm volatile(".reg .pred ddp_p0, ddp_p1, ddp_p2;")
#define DDP_MBAR_SPLIT(N)                                                                                                   \
    __device__ __forceinline__ void mbar_test_p##N(uint64_t *bar, uint32_t parity) {                                        \
        asm volatile("mbarrier.test_wait.parity.shared::cta.b64 ddp_p" #N ", [%0], %1;" ::"r"(smem_u32(bar)), "r"(parity)   \
                     : "memory");                                                                                           \
    }                                                                                                                       \
    __device__ __forceinline__ void mbar_finish_p##N(uint64_t *bar, uint32_t parity) {                                      \
        asm volatile(                                                                                                       \
            "{\n\t"                                                                                                         \
            "@ddp_p" #N " bra D_%=;\n\t"                                                                                    \
            "W_%=:\n\t"                                                                                                     \
            "mbarrier.try_wait.parity.shared::cta.b64 ddp_p" #N ", [%0], %1;\n\t"                                           \
            "@!ddp_p" #N " bra W_%=;\n\t"                                                                                   \
            "D_%=:\n\t}\n" ::"r"(smem_u32(bar)),                                                                           \
            "r"(parity)                                                                                                     \
            : "memory");                                                                                                    \
    }
DDP_MBAR_SPLIT(0)
DDP_MBAR_SPLIT(1)
DDP_MBAR_SPLIT(2)
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_alloc(uint32_t *dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, bf16 inputs, fp32 accumulate, both operands K-major
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// Same with the descriptors given as their low words (start address >> 4 | LBO >> 4 << 16); the high word is the
// constant SBO = 128 B (8 x 16 B core-matrix rows) | descriptor version 1, so advancing along K is one 32-bit add.
constexpr uint32_t DESC_HI = 8u | (1u << 14);
__device__ __forceinline__ void umma_bf16_lo(uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "mov.b64 da, {%1, %5};\n\t"
        "mov.b64 db, {%2, %5};\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, p;\n\t}\n" ::"r"(tmem_d),
        "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accumulate), "r"(DESC_HI)
        : "memory");
}
// A operand from tensor memory (lane = row, column c = packed bf16 pair k = 2c, 2c + 1): no shared-memory read of A,
// which in the SS form costs ~43 exposed cycles per MMA (profiles/r1_umma_microbench.txt)
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint32_t b_lo, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 db;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "mov.b64 db, {%2, %5};\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], db, %3, p;\n\t}\n" ::"r"(tmem_d),
        "r"(tmem_a), "r"(b_lo), "r"(idesc), "r"(accumulate), "r"(DESC_HI)
        : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]), "r"(r[1]),
                 "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
                 : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// One lane of the (converged) warp: the tcgen05 / TMA issue paths run warp-uniform and only the instruction itself
// is predicated, which keeps descriptors in uniform registers instead of per-lane broadcasts.
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred P;\n\t"
        "elect.sync _|P, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, P;\n\t}\n"
        : "=r"(pred));
    return pred != 0;
}
// no-swizzle K-major shared-memory descriptor: 8x(16 B) core matrices, LBO = stride between the two
// K-chunks of one MMA, SBO = stride between 8-row groups (cute::UMMA::SmemDescriptor, version 1)
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((addr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;
    return d;
}
__device__ __forceinline__ uint32_t instr_desc(int n) {
    // c=f32 (1<<4), a=bf16 (1<<7), b=bf16 (1<<10), K-major A and B, N>>3 at bit 17, M>>4 at bit 24
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(TILE_M >> 4) << 24);
}
// Asynchronous TMEM load of 16 columns (this thread's lane): the registers are valid only after tmem_wait16(v).
__device__ __forceinline__ void tmem_ld16_async(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
// tcgen05.wait::ld with the destination registers as in/out operands, so no consumer can be scheduled above it
__device__ __forceinline__ void tmem_wait16(uint32_t (&r)[16]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]),
                   "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
                 :
                 : "memory");
}
__device__ __forceinline__ void tmem_ld4_async(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                 : "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ void tmem_ld8_async(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ void red_add_v2(float *p, float a, float b) {
    asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(p), "f"(a), "f"(b) : "memory");
}
__device__ __forceinline__ void red_add_v4(float *p, float a, float b, float c, float d) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
// sum[0..N) += acc[0..N): 16-byte vector reductions when the row is 16-byte aligned, 8-byte ones otherwise (N even,
// rows always 8-byte aligned: f_out and every block offset are even)
template <int N, int NA>
__device__ __forceinline__ void red_row(float *dst, const float (&acc)[NA]) {
    static_assert(N % 2 == 0 && N <= NA, "even block widths only");
    if ((reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
#pragma unroll
        for (int o = 0; o + 4 <= N; o += 4) red_add_v4(dst + o, acc[o], acc[o + 1], acc[o + 2], acc[o + 3]);
        if (N % 4) red_add_v2(dst + N - 2, acc[N - 2], acc[N - 1]);
    } else {
#pragma unroll
        for (int o = 0; o < N; o += 2) red_add_v2(dst + o, acc[o], acc[o + 1]);
    }
}

// Deterministic mode (ddp_tpconv_umma*_fixed): the same pre-reduced partial sums, each converted to int64 fixed point
// (DDP_ACC_FIXED_SHIFT) and added with a 64-bit integer reduction -- associative, so the order in which CTAs, the two
// epilogue warpgroups and the split work items land does not show.  There is no vector form of red.add.u64: N
// reductions instead of N / 4.  dst is the row's first int64.
__device__ __forceinline__ void red_add_u64(unsigned long long *p, unsigned long long v) {
    asm volatile("red.global.add.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
template <int N, int NA>
__device__ __forceinline__ void red_row_fixed(unsigned long long *dst, const float (&acc)[NA], uint32_t *status) {
    static_assert(N <= NA, "block wider than the accumulator");
#pragma unroll
    for (int o = 0; o < N; ++o) red_add_u64(dst + o, ddp_to_fixed(acc[o], status));
}
// sum row of an output block: fp32 vector reductions, or fixed point in the deterministic mode
template <int N, bool FIXED, int NA>
__device__ __forceinline__ void flush_row(float *sum, size_t off, const float (&acc)[NA], uint32_t *status) {
    if constexpr (FIXED) red_row_fixed<N>(reinterpret_cast<unsigned long long *>(sum) + off, acc, status);
    else red_row<N>(sum + off, acc);
}

// Warp-level segmented inclusive scan of the output block over runs of consecutive edges with the same aggregation
// node (off = position of the lane inside its run): afterwards the last lane of every run holds the run's sum and is
// the only one that issues the atomics.  Edge lists whose aggregation side is sorted (receptor graph, ligand side of
// the cross edges, residue side of the atom-residue edges) have runs of 8 - 100 edges: 32 lanes adding to the SAME
// address serialise in the L2 atomic unit, the scan replaces them with log2(run) shuffle steps and one vector atomic.
template <int N, int NA>
__device__ __forceinline__ void seg_scan(float (&acc)[NA], int off, int nsteps) {
#pragma unroll 1
    for (int st = 0, d = 1; st < nsteps; ++st, d <<= 1) {
#pragma unroll
        for (int o = 0; o < N; ++o) {
            const float v = __shfl_up_sync(0xffffffffu, acc[o], d);
            if (off >= d) acc[o] += v;
        }
    }
}

__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
    __nv_bfloat162 t = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t *>(&t);
}

// ------------------------------------------------------------------------------------------ kernel
// NS scalar multiplicity, NV vector multiplicity, KS padded width of one A source block (>= NS + 1).
// K extent of one TMA slab / mbarrier round trip: 4 MMAs per wait amortise the issue-side latencies while the ring
// still holds ~2 weight tiles in flight (whole-tile slabs with 2 slots measured slower: the first MMA of a tile then
// waits for all of its 72 KB).
__host__ __device__ constexpr int stage_k_of(int ks, bool split) { return ks == 64 ? (split ? 32 : 64) : (split ? 16 : 32); }
// Tile shapes.  TS variant (hidden activations as a TMEM-resident A operand, single-pass bf16 only): a scalar tile
// covers ROWS_S basis rows x NS outputs padded to N = 192; TMEM holds two such fp32 accumulators next to the bf16
// hidden activations (2 x 208 + 96 columns = 512).  SS variant (A from shared memory; always used by the split mode):
// N = 240 scalar tiles, two 256-column accumulators.  A vector tile covers up to 2 NV basis rows x NV outputs, which
// the epilogue reads in two passes of NV rows.
// Measured on B200 (3dpf batch of 20, W = 10000 layers): SS 1.24 PFLOP/s, TS 1.04 PFLOP/s.  TS issues faster MMAs
// (106 vs 148 cycles) but its smaller tiles pay the per-tile hand-over (~500 cycles on both the issue and the epilogue
// side) more often and leave the tensor pipe idle in between, whereas in SS mode the exposed A-operand read hides
// those gaps.  TS stays selectable (-DDDP_UMMA_TS=1) for further work on the hand-over.
#ifndef DDP_UMMA_TS
#define DDP_UMMA_TS 0
#endif
#ifndef DDP_UMMA_DUAL
#define DDP_UMMA_DUAL 1
#endif
// DDP_UMMA_TOKEN = 1: the two issuers hand an issue-order token back and forth, so tiles reach the tensor pipe in tile
// order.  The token is REQUIRED for correctness with a ring shorter than two tiles' slabs (4 slots, 3 slabs per tile in the
// big-model configuration), not only an ordering nicety: an issuer that skips the other issuer's tile tests slot s for
// fill F while fill F-1 of s is one of the OTHER issuer's slabs, and bulk copies that are in flight together may land out
// of order (one misses in L2, a later one hits).  If that foreign slab is still in the air the parity test passes on the
// stale phase; the MMAs read a slot that is being written, their commit frees it early and the producer's
// mbarrier.arrive.expect_tx hits a barrier whose previous phase is still pending -> "Warp Illegal Instruction" at that
// SYNCS.ARRIVE.TRANS64 (cuda-gdb, profiles/r2_token0_rootcause.txt; seen only with two conv kernels in flight on two
// streams, where L2 contention reorders the copies; compute-sanitizer memcheck / synccheck / racecheck are clean for both
// builds).  The token is released after an issuer has ISSUED its tile -- so after it has seen every slab of that tile
// land -- and awaited before the first non-blocking parity test of the next tile, which closes the hole.
// tests/test_umma_protocol_model.py reproduces both the failure (no token, out-of-order landing) and the fix.
// 0 is a debug switch only.
#ifndef DDP_UMMA_TOKEN
#define DDP_UMMA_TOKEN 1
#endif
#ifndef DDP_UMMA_SEGSCAN
#define DDP_UMMA_SEGSCAN 1
#endif
// Diagnostic only (wrong results): 2 = full epilogue (default); 1 = TMEM loads kept, tensor-product FMAs skipped -- "what
// would the launch cost if the CUDA-core part of the epilogue were free" (profiles/r2_conv_energy_diag.txt).
#ifndef DDP_DIAG_EPI
#define DDP_DIAG_EPI 2
#endif
__host__ __device__ constexpr bool use_ts(bool split) { return DDP_UMMA_TS != 0 && !split; }
__host__ __device__ constexpr int rows_scalar(int ns, bool ts) { return (ts ? 192 : 240) / ns; }
__host__ __device__ constexpr int ncol_scalar(int ns, bool ts) { return (rows_scalar(ns, ts) * ns + 15) / 16 * 16; }
__host__ __device__ constexpr int rows_vector(int nv) { return 2 * nv; }
__host__ __device__ constexpr int ncol_vector(int nv, int n_rows) { return (n_rows * nv + 15) / 16 * 16; }

constexpr int MAX_JOBS = 9;
constexpr int N_EPI = 128, N_GATHER = 64, N_THREADS = 384;   // N_EPI: threads of ONE epilogue warpgroup; N_GATHER: arrivals that complete an a_ready phase
// Registers per thread after the setmaxnreg hand-over: 384 threads start with 168 (64512 in total); the producer / issuer /
// gather warpgroup keeps REGS_AUX, each epilogue warpgroup grows to REGS_EPI (128 * 104 + 256 * 200 = 64512).
constexpr int REGS_AUX = 104, REGS_EPI = 200;
static_assert(128 * REGS_AUX + 2 * N_EPI * REGS_EPI <= N_THREADS * 168, "register hand-over exceeds the CTA's allocation");

// One fused convolution of a grouped launch.  All jobs of a launch share irreps (tile table, f_in, f_out).
struct Job {
    const uint8_t *image;
    ddp_tpconv_edges_t ed;
    float *sum;
};
struct Jobs {
    int32_t n, f_in, f_out;
    long long *trace;     // optional timing trace of CTA 0 (ddp_tpconv_umma_set_trace), NULL in production
    Job job[MAX_JOBS];
    uint32_t *status;     // sticky status word of the deterministic mode (FIXED kernels only; after job[] so that the
                          // parameter offsets of the default kernels stay where they were)
};
[[maybe_unused]] constexpr int TRACE_EVENTS = 8, TRACE_TILES = 256;
// trace[(role * TRACE_TILES + tile iteration) * TRACE_EVENTS + event] = clock64 (CTA 0, one lane per role)
// Compiled in only with -DDDP_UMMA_TRACE (scripts/umma_trace.py builds such a library): the hooks sit in the per-tile
// loops of the issue and epilogue warps and cost ~5 % of the epilogue's instructions even when the pointer is NULL.
__device__ __forceinline__ void trace_ev(long long *trace, int role, int iter, int ev) {
#ifdef DDP_UMMA_TRACE
    if (trace != nullptr && blockIdx.x == 0 && iter < TRACE_TILES) trace[(role * TRACE_TILES + iter) * TRACE_EVENTS + ev] = clock64();
#else
    (void)trace; (void)role; (void)iter; (void)ev;
#endif
}

template <int NS, int NV, int KS, bool SPLIT>
struct Cfg {
    static constexpr int KP = 3 * KS;                       // padded K of both GEMMs (and padded hidden width N1)
    static constexpr int N1 = KP;
    static constexpr bool TS = use_ts(SPLIT);               // hidden activations as a TMEM-resident A operand
    static constexpr int ROWS_S = rows_scalar(NS, TS);
    static constexpr int NVAL_S = ROWS_S * NS;              // weight columns of a scalar tile
    static constexpr int NCOL_S = ncol_scalar(NS, TS);      // ... padded to the UMMA N granularity
    static constexpr int ROWS_V = rows_vector(NV);
    static constexpr int PASS_COLS = NV * NV;               // weight columns the epilogue handles per pass (NV rows)
    static constexpr int NCOL_V = ncol_vector(NV, ROWS_V);
    static constexpr int NCOL_MAX = (NCOL_S > N1 ? (NCOL_S > NCOL_V ? NCOL_S : NCOL_V) : (N1 > NCOL_V ? N1 : NCOL_V));
    static constexpr int ACC_STRIDE = TS ? 208 : 256;       // TMEM columns between the two accumulators
    static constexpr int H_COL = 2 * ACC_STRIDE;            // TS: first TMEM column of the hidden activations (KP / 2 columns)
    static constexpr int STAGE_K = stage_k_of(KS, SPLIT);
    static constexpr int STAGE_BYTES = NCOL_MAX * STAGE_K * 2 * (SPLIT ? 2 : 1);
    static constexpr int A_BYTES = TILE_M * KP * 2;         // one bf16 A image
    // A operand buffers in shared memory.  TS: one (free again as soon as GEMM1 has run); SS: two, so that the next
    // edge tile is gathered under the current GEMM2 (split mode: one, its hi + lo images are already 96 KB)
    static constexpr int NBUF = (TS || SPLIT) ? 1 : 2;
    static constexpr int A_TOTAL = A_BYTES * (SPLIT ? 2 : 1) * NBUF;
    static constexpr int MAX_TILES = 64;
    static constexpr int FIXED = 1024 + A_TOTAL + MAX_TILES * (int)sizeof(TileDesc) + 1024;
    static constexpr int STAGES_FIT = (220 * 1024 - FIXED) / STAGE_BYTES;
    static constexpr int STAGES = STAGES_FIT > 12 ? 12 : STAGES_FIT;
    static constexpr size_t SMEM = (size_t)FIXED + (size_t)STAGES * STAGE_BYTES;
    static constexpr bool DUAL = DDP_UMMA_DUAL != 0 && STAGES >= KP / STAGE_K + 1;   // two MMA issuers (see the issue loop)
    static constexpr int XN_RAW = 3 * NV > 3 * ROWS_S ? 3 * NV : 3 * ROWS_S;   // floats of x one tile reads (x (x) s1 tiles: 2 NV,
    static constexpr int XN = XN_RAW + (XN_RAW & 1);                              //  stride-3 kinds: NV or ROWS_S rows of 3)
    static_assert(N1 % 16 == 0 && NCOL_MAX <= ACC_STRIDE && (TS ? H_COL + KP / 2 : H_COL) <= 512, "UMMA N / TMEM budget");
    static_assert(KS >= NS + 1 && KP % STAGE_K == 0, "K padding");
    static_assert(STAGES >= 2, "weight ring too small");
    static_assert(XN % 2 == 0, "x prefetch registers are loaded in pairs");
};

// TMEM accumulator of slot tt of an item with nt weight tiles (tt = -1: GEMM1, always accumulator 0).  The weight tiles
// alternate such that the LAST one sits in accumulator 1: accumulator 0 is then free one tile earlier, and the next
// item's GEMM1 runs under the last tile's MMAs / epilogue instead of after them.  For even nt that puts GEMM1 and
// tile 0 back to back in accumulator 0 (tile 0 has to wait for the hidden activations anyway).
__device__ __forceinline__ uint32_t acc_of(int tt, int nt) { return tt < 0 ? 0u : (uint32_t)(tt + nt) & 1u; }

// Map the g-th 128-edge tile of the launch to (job, tile inside the job); pref = exclusive prefix of tile counts.
__device__ __forceinline__ void locate(const int *pref, int n_jobs, int g, int &job, int &et) {
    int j = 0;
    while (j + 1 < n_jobs && g >= pref[j + 1]) ++j;
    job = j;
    et = g - pref[j];
}

// Work items.  Edge tiles are dealt round-robin to the CTAs; the last, partial round (R = n_etiles mod grid tiles for
// grid CTAs) would leave most SMs idle for a whole tile time, so each of its edge tiles is split `k` ways along the
// weight tiles (contiguous ranges of equal MMA cost): every part redoes the cheap gather + GEMM1 and adds its partial
// sums with the same atomics.  Item w < n_full: edge tile w, all weight tiles; else edge tile n_full + (w - n_full) / k,
// weight tiles [split[p], split[p + 1]) with p = (w - n_full) % k.
constexpr int SPLIT_MAX = 8;
struct Work {
    int n_items, n_full, k;
    int split[SPLIT_MAX + 1];
};
__device__ __forceinline__ void work_item(const Work &wk, int w, int n_tiles, int &g, int &t0, int &t1) {
    if (w < wk.n_full) { g = w; t0 = 0; t1 = n_tiles; return; }
    const int idx = w - wk.n_full;
    g = wk.n_full + idx / wk.k;
    const int p = idx % wk.k;
    t0 = wk.split[p];
    t1 = wk.split[p + 1];
}

// Issue the global loads of the gathered node features one weight tile reads (n_fl floats from xg): pairs when the
// offset is even (rows are 8-byte aligned), single floats otherwise.  Predicated, branch-free.
template <int XN>
__device__ __forceinline__ void x_prefetch(const float *xg, int n_fl, float (&xn)[XN]) {
    if ((reinterpret_cast<uintptr_t>(xg) & 7) == 0) {
#pragma unroll
        for (int j = 0; j < XN / 2; ++j)
            if (2 * j < n_fl) {
                const float2 v = __ldg(reinterpret_cast<const float2 *>(xg) + j);
                xn[2 * j] = v.x; xn[2 * j + 1] = v.y;
            }
    } else {
#pragma unroll
        for (int j = 0; j < XN; ++j)
            if (j < n_fl) xn[j] = __ldg(xg + j);
    }
}

// Same, for a compile-time count (the common case: full tiles): N / 2 unpredicated 8-byte loads.
template <int N, int XN>
__device__ __forceinline__ void x_prefetch_n(const float *xg, float (&xn)[XN]) {
    static_assert(N % 2 == 0 && N <= XN, "pairs");
#pragma unroll
    for (int j = 0; j < N / 2; ++j) {
        const float2 v = __ldg(reinterpret_cast<const float2 *>(xg) + j);
        xn[2 * j] = v.x; xn[2 * j + 1] = v.y;
    }
}
// Node features of the weight tile described by tdw: full tiles of every kind take the unpredicated path.
template <int NS, int NV, int ROWS_S, int XN>
__device__ __forceinline__ void x_prefetch_tile(const float *xg_row, const uint4 &tdw, int f_in, float (&xn)[XN]) {
    const int kind = (int)((tdw.x >> 16) & 0xffu), n_rows = (int)(tdw.x >> 24), x_off = (int)(tdw.z & 0xffffu);
    const float *xg = xg_row + x_off;
    constexpr int N0 = ROWS_S + (ROWS_S & 1), N1 = 3 * ROWS_S + (ROWS_S & 1), N2 = 2 * NV, N3 = 3 * NV + (NV & 1);
    const int full = kind == 0 ? N0 : (kind == 1 ? N1 : (kind == 2 ? N2 : N3));
    const bool fast = (reinterpret_cast<uintptr_t>(xg) & 7) == 0 && x_off + full <= f_in;   // stays inside the node's row
    if (fast && kind == 0) x_prefetch_n<N0, XN>(xg, xn);
    else if (fast && kind == 1) x_prefetch_n<N1, XN>(xg, xn);
    else if (fast && kind == 2) x_prefetch_n<N2, XN>(xg, xn);
    else if (fast) x_prefetch_n<N3, XN>(xg, xn);
    else x_prefetch<XN>(xg, n_rows * ((kind == 0 || kind == 2) ? 1 : 3), xn);
}

// Stage ROWS rows per lane (row0 + lane + 32 h) of the A operand of edge tile `et`: [emb | p1 | p2] as bf16 (constant
// one in slot NS of source 0), written in UMMA core-matrix order (hi image, plus the lo image in split mode).  The
// index loads are issued before the wait for the buffer, the feature loads after it.
template <int NS, int KS, bool SPLIT, int ROWS>
__device__ __forceinline__ void gather_rows(const ddp_tpconv_edges_t &ed, int n_edges, int et, int row0, int lane, uint8_t *a_hi,
                                            uint8_t *a_lo, uint64_t *free_bar, uint32_t free_parity) {
    const float *srcs[ROWS][3];
#pragma unroll
    for (int h = 0; h < ROWS; ++h) {
        const int e = et * TILE_M + row0 + lane + h * 32;
        const bool valid = e < n_edges;
        srcs[h][0] = valid ? ed.emb + (size_t)e * NS : nullptr;
        srcs[h][1] = valid ? ed.p1 + (size_t)__ldg(ed.i1 + e) * ed.ld1 : nullptr;
        srcs[h][2] = valid ? ed.p2 + (size_t)__ldg(ed.i2 + e) * ed.ld2 : nullptr;
    }
#ifdef DDP_UMMA_SPIN
    mbar_wait(free_bar, free_parity);
#else
    mbar_wait_relaxed<500>(free_bar, free_parity);
#endif
#pragma unroll
    for (int h = 0; h < ROWS; ++h) {
        const int r = row0 + lane + h * 32;
        const uint32_t a_row_off = (uint32_t)((r >> 3) * 128 + (r & 7) * 16);
#pragma unroll
        for (int s = 0; s < 3; ++s) {
            const float *sp = srcs[h][s];
            const bool v4 = (s == 0) ? (NS % 4 == 0) : (((s == 1 ? ed.ld1 : ed.ld2) & 3) == 0);
#pragma unroll
            for (int c8 = 0; c8 < KS / 8; ++c8) {
                float v[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) v[q] = 0.f;
                if (sp != nullptr) {
                    if (v4 && NS % 4 == 0) {
                        if (c8 * 8 < NS) {
                            const float4 f = __ldg(reinterpret_cast<const float4 *>(sp + c8 * 8));
                            v[0] = f.x; v[1] = f.y; v[2] = f.z; v[3] = f.w;
                        }
                        if (c8 * 8 + 4 < NS) {
                            const float4 f = __ldg(reinterpret_cast<const float4 *>(sp + c8 * 8 + 4));
                            v[4] = f.x; v[5] = f.y; v[6] = f.z; v[7] = f.w;
                        }
                    } else {
#pragma unroll
                        for (int q = 0; q < 8; ++q)
                            if (c8 * 8 + q < NS) v[q] = __ldg(sp + c8 * 8 + q);
                    }
                }
                if (s == 0 && NS / 8 == c8) v[NS % 8] = 1.f;
                uint4 hi;
                hi.x = pack_bf16x2(v[0], v[1]); hi.y = pack_bf16x2(v[2], v[3]);
                hi.z = pack_bf16x2(v[4], v[5]); hi.w = pack_bf16x2(v[6], v[7]);
                const uint32_t off = (uint32_t)((s * (KS / 8) + c8) * (TILE_M * 16)) + a_row_off;
                *reinterpret_cast<uint4 *>(a_hi + off) = hi;
                if (SPLIT) {
                    float w[8];
#pragma unroll
                    for (int q = 0; q < 8; ++q) w[q] = v[q] - __bfloat162float(__float2bfloat16_rn(v[q]));
                    uint4 lo;
                    lo.x = pack_bf16x2(w[0], w[1]); lo.y = pack_bf16x2(w[2], w[3]);
                    lo.z = pack_bf16x2(w[4], w[5]); lo.w = pack_bf16x2(w[6], w[7]);
                    *reinterpret_cast<uint4 *>(a_lo + off) = lo;
                }
            }
        }
    }
    fence_proxy_async();
}

// L2: the edge harmonics have 9 components (sh_lmax = 2, e3nn FullyConnectedTensorProduct trunk convs) and kind-5 tiles
// exist; a separate instantiation so that the sh_lmax = 1 kernel keeps its register allocation.
template <int NS, int NV, int KS, bool SPLIT, bool L2, bool FIXED>
__global__ void __launch_bounds__(N_THREADS, 1)
tpconv_umma_kernel(const __grid_constant__ Jobs jobs) {
    using C = Cfg<NS, NV, KS, SPLIT>;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    // carve (everything 128 B aligned)
    uint8_t *p = smem_raw;
    uint8_t *a_base = p;                   p += C::A_TOTAL;            // [NBUF][hi (, lo)]
    uint8_t *ring = p;                     p += (size_t)C::STAGES * C::STAGE_BYTES;
    TileDesc *tiles = reinterpret_cast<TileDesc *>(p); p += C::MAX_TILES * sizeof(TileDesc);
    uint64_t *bars = reinterpret_cast<uint64_t *>(p);
    uint64_t *full = bars, *empty = bars + C::STAGES;
    uint64_t *tmem_full = bars + 2 * C::STAGES, *tmem_empty = tmem_full + 2;
    uint64_t *a_ready = tmem_empty + 2, *a_free = a_ready + 2, *h_ready = a_free + 2;
    uint64_t *tok = h_ready + 1;                                        // [2] issue-order token of the two MMA issuers
    uint32_t *tmem_base_smem = reinterpret_cast<uint32_t *>(tok + 2);
    int *pref = reinterpret_cast<int *>(tmem_base_smem + 2);            // [MAX_JOBS + 1]
    Work *work = reinterpret_cast<Work *>(pref + MAX_JOBS + 1);
    uint32_t *tile_off = reinterpret_cast<uint32_t *>(work + 1);        // [MAX_TILES + 1] byte offset of every tile's slabs
    int *cum = reinterpret_cast<int *>(tile_off + C::MAX_TILES + 1);    // [MAX_TILES + 1] MMA cost prefix (set-up only)

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_jobs = jobs.n, f_in = jobs.f_in, f_out = jobs.f_out;
    const Header *hdr = reinterpret_cast<const Header *>(jobs.job[0].image);
    const int n_tiles = hdr->n_tiles;

    for (int i = threadIdx.x; i < n_tiles * (int)(sizeof(TileDesc) / 4); i += blockDim.x)
        reinterpret_cast<uint32_t *>(tiles)[i] = reinterpret_cast<const uint32_t *>(jobs.job[0].image + hdr->tiles_off)[i];
    if (threadIdx.x == 0) {
        for (int s = 0; s < C::STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        for (int b = 0; b < 2; ++b) {
            mbar_init(&tmem_full[b], 1); mbar_init(&tmem_empty[b], N_EPI);
            mbar_init(&a_ready[b], N_GATHER); mbar_init(&a_free[b], (C::TS || !C::DUAL) ? 1 : 2);
        }
        mbar_init(h_ready, N_EPI);
        mbar_init(&tok[0], 1); mbar_init(&tok[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // tile counts of the jobs: one thread per job fetches its live edge count (independent loads), warp 7 scans them
    if (warp == 7) {
        int nt = 0;
        if (lane < n_jobs) nt = (min(__ldg(jobs.job[lane].ed.n_edges_dev), jobs.job[lane].ed.edge_cap) + TILE_M - 1) / TILE_M;
        int incl = nt;
#pragma unroll
        for (int o = 1; o < 16; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        if (lane < n_jobs) pref[lane] = incl - nt;
        if (lane == n_jobs - 1) pref[n_jobs] = incl;
    }
    if (warp == 5) tmem_alloc(tmem_base_smem, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_base_smem;
    const int slabs_off = (int)hdr->slabs_off;
    if (threadIdx.x == 0) {
        // slab byte offsets (W1 slabs first, then every weight tile) and MMA cost prefix (cost ~ UMMA N + exposed A read)
        uint32_t off = (uint32_t)slab_bytes(C::N1, C::STAGE_K, SPLIT) * (C::KP / C::STAGE_K);
        cum[0] = 0;                                                         // (shared memory: a stack array would be cold DRAM round trips)
        for (int t = 0; t < n_tiles; ++t) {
            tile_off[t] = off;
            off += (uint32_t)slab_bytes(tiles[t].n_cols, C::STAGE_K, SPLIT) * (C::KP / C::STAGE_K);
            cum[t + 1] = cum[t] + tiles[t].n_cols + 86;
        }
        tile_off[n_tiles] = off;
        const int total = pref[n_jobs], G = (int)gridDim.x;
        const int R = total % G;
        int k = 1;
        if (R > 0) k = min(min(SPLIT_MAX, G / R), n_tiles);
        work->n_full = k > 1 ? total - R : total;
        work->k = k;
        work->n_items = work->n_full + (k > 1 ? R * k : 0);
        int t = 0;
        for (int p = 0; p <= k; ++p) {
            const int target = (int)((long long)cum[n_tiles] * p / k);
            while (t < n_tiles && cum[t] < target) ++t;
            work->split[p] = p == k ? n_tiles : t;
        }
        for (int p = 1; p < k; ++p)                                         // every part keeps at least one tile
            work->split[p] = min(max(work->split[p], work->split[p - 1] + 1), n_tiles - (k - p));
    }
    __syncthreads();
    const Work &wk = *work;
    const int n_items = wk.n_items;

    // register hand-over (warpgroup-wide; each setmaxnreg sits at the head of the code it governs so that ptxas allocates
    // the two sides separately)
    if (warp >= 4 && warp < 8) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_AUX));
    if (C::DUAL && warp == 7 && (int)blockIdx.x < n_items) {
        // rows 64..127 of the CTA's first edge tile (then this warp turns MMA issuer)
        int g, t0, t1, job, et;
        work_item(wk, blockIdx.x, n_tiles, g, t0, t1);
        locate(pref, n_jobs, g, job, et);
        const ddp_tpconv_edges_t &ed = jobs.job[job].ed;
        gather_rows<NS, KS, SPLIT, 2>(ed, min(*ed.n_edges_dev, ed.edge_cap), et, 64, lane, a_base, a_base + C::A_BYTES, &a_free[0], 1u);
        mbar_arrive(&a_ready[0]);
    }
    if (warp == 4) {
        // =============================== TMA producer (warp-uniform, one elected lane issues) =====
        uint32_t stage = 0, phase = 0;
        for (int w = blockIdx.x; w < n_items; w += gridDim.x) {
            int g, t0, t1, job, et;
            work_item(wk, w, n_tiles, g, t0, t1);
            locate(pref, n_jobs, g, job, et);
            const uint8_t *base = jobs.job[job].image + slabs_off;
            for (int tt = -1; tt < t1 - t0; ++tt) {
                const int t = tt < 0 ? -1 : t0 + tt;
                const uint8_t *src = t < 0 ? base : base + tile_off[t];
                const int ncol = (t < 0) ? C::N1 : tiles[t].n_cols;
                const uint32_t bytes = slab_bytes(ncol, C::STAGE_K, SPLIT);
#pragma unroll 1
                for (int ks = 0; ks < C::KP / C::STAGE_K; ++ks) {
                    DDP_WAIT_RELAXED(0, &empty[stage], phase ^ 1, 1, w, tt * 8 + ks);
                    if (elect_one()) {
                        mbar_expect_tx(&full[stage], bytes);
                        bulk_g2s(ring + (size_t)stage * C::STAGE_BYTES, src, bytes, &full[stage]);
                    }
                    __syncwarp();
                    src += bytes;
                    if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 5 || (warp == 7 && C::DUAL)) {
        // =============================== MMA issuers (warp-uniform, one elected lane issues) ======
        // Two issuers, one per accumulator: warp 5 owns accumulator 0 (GEMM1 and the odd weight tiles), warp 7
        // accumulator 1 (the even weight tiles).  tcgen05.mma issue blocks while the tensor pipe's short queue is
        // full, so a single issuer exposes everything it does between two tiles (barrier round trips, descriptor
        // set-up: ~270 cycles per 1450-cycle tile in profiles/r1_umma_timeline_cta0_layer3_v17.txt); with two, one is
        // already parked on the queue with its next tile while the other finishes the current one.  Tiles of the two
        // accumulators are independent, so the order in which the pipe interleaves them does not matter; every slab
        // stage, accumulator and barrier phase has exactly one owner.  Inside a tile the test of the next K group's
        // slab is split-phase (started before the group is issued, consumed after it).
        // (Configurations whose ring is shorter than one tile's slabs + 1 keep a single issuer: an issuer that skips a
        // whole foreign tile could otherwise wait on a slab whose slot is still two fills behind -- parity aliasing.)
        DDP_DECLARE_TEST_PREDS();
        const uint32_t me = warp == 5 ? 0u : 1u;
        uint32_t stage = 0, phase = 0;
        uint32_t te_phase = 0;               // bit b: parity to wait on tmem_empty[b]
        uint32_t hr_phase = 0;
        uint32_t tok_phase = 0;              // parity of the other issuer's next "tile issued" token
        int tok_pending = 0;                 // foreign tiles skipped since this issuer's last tile
        int it = 0;
        constexpr int NG = C::KP / C::STAGE_K;
        int titer = 0;
        for (int w = blockIdx.x; w < n_items; w += gridDim.x, ++it) {
            int g, t0, t1;
            work_item(wk, w, n_tiles, g, t0, t1);
            const int nt = t1 - t0;
            const int ab = it % C::NBUF;
            const uint32_t a_hi_addr = smem_u32(a_base + (size_t)ab * C::A_BYTES * (SPLIT ? 2 : 1));
            // descriptor low words: A has LBO = 128 rows x 16 B between the two K chunks of one MMA
            const uint32_t a_hi_lo = ((a_hi_addr >> 4) & 0x3FFFu) | ((uint32_t)(TILE_M * 16 >> 4) << 16);
            const uint32_t a_lo_lo = (((a_hi_addr + C::A_BYTES) >> 4) & 0x3FFFu) | ((uint32_t)(TILE_M * 16 >> 4) << 16);
            for (int tt = -1; tt < nt; ++tt, ++titer) {
                const uint32_t buf = acc_of(tt, nt);
                if (C::DUAL && buf != me) {                              // the other issuer's tile: only the ring position moves
#pragma unroll
                    for (int ks = 0; ks < NG; ++ks)
                        if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
                    ++tok_pending;
                    continue;
                }
                const int t = tt < 0 ? -1 : t0 + tt;                     // weight tile (-1: GEMM1)
                const uint32_t ncol = (t < 0) ? (uint32_t)C::N1 : (uint32_t)tiles[t].n_cols;
                const uint32_t d_tmem = tmem_base + buf * (uint32_t)C::ACC_STRIDE;
                const uint32_t idesc = instr_desc((int)ncol);
                // B: LBO = ncol rows x 16 B; one K = 16 step advances the start address by 2 * LBO
                const uint32_t b_lbo_word = ncol << 16;
                const uint32_t b_step = 2u * ncol;                      // (2 * ncol * 16 B) >> 4
                const bool ts = C::TS && t >= 0;                        // GEMM2 reads the hidden activations from TMEM
                // the A buffer is free once its last reader has run: GEMM1 (TS) / both issuers' last tiles (SS)
                const bool last_reader = C::TS ? tt < 0 : tt + (C::DUAL ? 2 : 1) >= nt;
                trace_ev(jobs.trace, 0, titer, 0);
                if (tt < 0) DDP_WAIT(&a_ready[ab], (uint32_t)(it / C::NBUF) & 1u, 2, it, tt);
                // the first GEMM2 tile this warp issues in the item needs the hidden activations (tile 0, and tile 1 where
                // it belongs to the other issuer); every warp toggles its phase once per item
                if (tt == 0 || (C::DUAL && tt == 1)) DDP_WAIT(h_ready, hr_phase, 3, it, tt);
                DDP_WAIT(&tmem_empty[buf], ((te_phase >> buf) & 1u) ^ 1u, 4, it, tt);
                te_phase ^= 1u << buf;
                DDP_WAIT(&full[stage], phase, 5, it, tt * 16 + (int)stage);
                if (C::DUAL && DDP_UMMA_TOKEN) {
                    // tiles are issued in tile order: everything above overlapped the other issuer's tile, only the
                    // first tcgen05.mma waits for its last one
                    // (one token per run of the other issuer's tiles: warp 5 owns GEMM1 and tile 0 of an even-length item
                    // back to back and signals only after the second)
                    if (tok_pending > 0) { DDP_WAIT(&tok[me ^ 1u], tok_phase, 6, it, tt); tok_phase ^= 1u; tok_pending = 0; }
                }
                tc_fence_after();
                trace_ev(jobs.trace, 0, titer, 1);
                trace_ev(jobs.trace, 0, titer, 2);
#pragma unroll
                for (int ks = 0; ks < NG; ++ks) {
                    // the slab of this group has landed (blocking wait above, or the finish of the previous group)
                    uint32_t ns_ = stage + 1, np_ = phase;
                    if (ns_ == C::STAGES) { ns_ = 0; np_ ^= 1; }
#ifndef DDP_UMMA_WATCHDOG
                    if (ks + 1 < NG) mbar_test_p0(&full[ns_], np_);
#endif
                    const uint32_t b_addr = smem_u32(ring + (size_t)stage * C::STAGE_BYTES);
                    const uint32_t b_lo0 = ((b_addr >> 4) & 0x3FFFu) | b_lbo_word;
                    const uint32_t a_k = (uint32_t)(ks * (C::STAGE_K / 8)) * (uint32_t)(TILE_M * 16 >> 4);
                    const uint32_t a_t = tmem_base + (uint32_t)C::H_COL + (uint32_t)(ks * (C::STAGE_K / 2));
                    if (elect_one()) {
#pragma unroll
                        for (int kk = 0; kk < C::STAGE_K / 16; ++kk) {
                            const uint32_t a_off = a_k + (uint32_t)(2 * kk) * (uint32_t)(TILE_M * 16 >> 4);
                            const uint32_t b_lo = b_lo0 + (uint32_t)kk * b_step;
                            if (ts) umma_bf16_ts(d_tmem, a_t + (uint32_t)(8 * kk), b_lo, idesc, (ks | kk) != 0);
                            else umma_bf16_lo(d_tmem, a_hi_lo + a_off, b_lo, idesc, (ks | kk) != 0);
                            if (SPLIT) {
                                const uint32_t bl_lo = b_lo + ((ncol * (uint32_t)C::STAGE_K * 2u) >> 4);
                                umma_bf16_lo(d_tmem, a_lo_lo + a_off, b_lo, idesc, 1);
                                umma_bf16_lo(d_tmem, a_hi_lo + a_off, bl_lo, idesc, 1);
                            }
                        }
                        umma_commit(&empty[stage]);
                        if (ks == NG - 1) {
                            umma_commit(&tmem_full[buf]);
                            if (last_reader) umma_commit(&a_free[ab]);
                            if (C::DUAL && DDP_UMMA_TOKEN && !(tt < 0 && acc_of(0, nt) == 0u)) mbar_arrive(&tok[me]);
                        }
                    }
                    __syncwarp();
#ifndef DDP_UMMA_WATCHDOG
                    if (ks + 1 < NG) { mbar_finish_p0(&full[ns_], np_); tc_fence_after(); }
#else
                    if (ks + 1 < NG) { DDP_WAIT(&full[ns_], np_, 11, it, tt * 16 + (int)ns_); tc_fence_after(); }
#endif
                    stage = ns_; phase = np_;
                }
                trace_ev(jobs.trace, 0, titer, 3);
            }
            hr_phase ^= 1u;
        }
    } else {
        // =============================== gather: A operand of the NEXT edge tile (warp 6; warp 7 too without DUAL) ===
        // Two-issuer configurations: warp 6 stages all 128 rows of every edge tile (four per lane) except the CTA's
        // first one, where warp 7 -- idle as an issuer until the first hidden activations exist -- has taken rows
        // 64..127 (see above) so that the launch does not start with a single warp's gather latency.  Single-issuer
        // configurations: warps 6 and 7 stage 64 rows each.  a_ready counts 64 arrivals either way.
        int it = 0;
        for (int w = blockIdx.x; w < n_items; w += gridDim.x, ++it) {
            int g, t0, t1, job, et;
            work_item(wk, w, n_tiles, g, t0, t1);
            locate(pref, n_jobs, g, job, et);
            const ddp_tpconv_edges_t &ed = jobs.job[job].ed;
            const int n_edges = min(*ed.n_edges_dev, ed.edge_cap);
            const int ab = it % C::NBUF;
            uint8_t *a_hi = a_base + (size_t)ab * C::A_BYTES * (SPLIT ? 2 : 1);
            uint8_t *a_lo = a_hi + C::A_BYTES;
            const uint32_t fpar = ((uint32_t)(it / C::NBUF) & 1u) ^ 1u;
            if (C::DUAL && it > 0) {
                gather_rows<NS, KS, SPLIT, 4>(ed, n_edges, et, 0, lane, a_hi, a_lo, &a_free[ab], fpar);
                mbar_arrive(&a_ready[ab]);
            } else {
                gather_rows<NS, KS, SPLIT, 2>(ed, n_edges, et, (warp - 6) * 64, lane, a_hi, a_lo, &a_free[ab], fpar);
            }
            mbar_arrive(&a_ready[ab]);
        }
    }
    } else {
        // =============================== epilogue warps: one warpgroup per accumulator ==============
        asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REGS_EPI));
        const uint32_t wg = (uint32_t)warp >> 3;         // accumulator this warpgroup reads (warps 0-3: 0, warps 8-11: 1)
        const int r = threadIdx.x & 127;                 // edge row = TMEM lane
        const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
        const bool tracer = r == 0;                      // trace role 1 + wg
        uint32_t tf_phase = 0;                           // parity to wait on tmem_full[wg] (warpgroup 0: GEMM1 results and tiles alike)
        const uint32_t a_row_off = (uint32_t)((r >> 3) * 128 + (r & 7) * 16);
        const uint32_t taddr = tmem_base + lane_base + wg * (uint32_t)C::ACC_STRIDE;
        int it = 0;
        // Warpgroup 0 only.  GEMM1 result -> ReLU -> hidden activations become the A operand of GEMM2 (TS: packed bf16 pairs
        // into tensor memory, column c of the lane = k 2c, 2c + 1; SS: hi (/ lo) images back into the shared-memory A buffer
        // in core-matrix order).  At an item boundary warpgroup 0's last own tile is the last but one of the item, and the next
        // item's GEMM1 is issued behind the last tile: the ~2400 cycles until its result exists take the warpgroup's last flush
        // and the next item's per-edge set-up (dependent global loads), so that after the conversion tile 0's epilogue is
        // ready when its MMAs are (profiles/r2_umma_timeline_*.txt).
        auto convert_hidden = [&](uint8_t *a_hi_, uint8_t *a_lo_, int it_) {
            if (tracer) trace_ev(jobs.trace, 1, it_ * (n_tiles + 1), 0);
            DDP_WAIT(&tmem_full[0], tf_phase, 8, it_, -1);
            tf_phase ^= 1u;
            tc_fence_after();
            if (tracer) trace_ev(jobs.trace, 1, it_ * (n_tiles + 1), 1);
            {
                uint32_t w[2][16];
                tmem_ld16_async(tmem_base + lane_base, w[0]);
#pragma unroll
                for (int c16 = 0; c16 < C::N1 / 16; ++c16) {
                    tmem_wait16(w[c16 & 1]);
                    if (c16 + 1 < C::N1 / 16) tmem_ld16_async(tmem_base + lane_base + (uint32_t)((c16 + 1) * 16), w[(c16 + 1) & 1]);
                    float v[16];
#pragma unroll
                    for (int q = 0; q < 16; ++q) v[q] = fmaxf(__uint_as_float(w[c16 & 1][q]), 0.f);
                    if (C::TS) {
                        uint32_t pk[8];
#pragma unroll
                        for (int q = 0; q < 8; ++q) pk[q] = pack_bf16x2(v[2 * q], v[2 * q + 1]);
                        tmem_st8(tmem_base + lane_base + (uint32_t)(C::H_COL + c16 * 8), pk);
                    } else {
#pragma unroll
                        for (int h8 = 0; h8 < 2; ++h8) {
                            uint4 hi;
                            hi.x = pack_bf16x2(v[8 * h8 + 0], v[8 * h8 + 1]); hi.y = pack_bf16x2(v[8 * h8 + 2], v[8 * h8 + 3]);
                            hi.z = pack_bf16x2(v[8 * h8 + 4], v[8 * h8 + 5]); hi.w = pack_bf16x2(v[8 * h8 + 6], v[8 * h8 + 7]);
                            const uint32_t off = (uint32_t)((c16 * 2 + h8) * (TILE_M * 16)) + a_row_off;
                            *reinterpret_cast<uint4 *>(a_hi_ + off) = hi;
                            if (SPLIT) {
                                float u[8];
#pragma unroll
                                for (int q = 0; q < 8; ++q) u[q] = v[8 * h8 + q] - __bfloat162float(__float2bfloat16_rn(v[8 * h8 + q]));
                                uint4 lo;
                                lo.x = pack_bf16x2(u[0], u[1]); lo.y = pack_bf16x2(u[2], u[3]);
                                lo.z = pack_bf16x2(u[4], u[5]); lo.w = pack_bf16x2(u[6], u[7]);
                                *reinterpret_cast<uint4 *>(a_lo_ + off) = lo;
                            }
                        }
                    }
                }
            }
            if (tracer) trace_ev(jobs.trace, 1, it_ * (n_tiles + 1), 3);
            if (C::TS) tmem_wait_st();
            tc_fence_before();
            if (!C::TS) fence_proxy_async();
            mbar_arrive(h_ready);
            mbar_arrive(&tmem_empty[0]);
            if (tracer) trace_ev(jobs.trace, 1, it_ * (n_tiles + 1), 2);
        };
        // First-level per-edge loads of an item (live edge count, aggregation node, gathered node, edge harmonics): issued one
        // item ahead -- for the CTA's first item here, for item i + 1 at the top of item i -- so that at an item boundary only
        // the loads that depend on them (in-degree, node features) remain, and those run under the hidden conversion.  The
        // chain count -> agg -> degree / gather -> features was ~6000 cycles of exposed L2 latency per boundary
        // (profiles/r2_umma_timeline_*.txt).  Rows past the live count read allocated but meaningless entries (e < edge_cap).
        int nx_ne = 0, nx_agg = 0, nx_gather = 0;
        float nx_s0 = 0.f, nx_s1x = 0.f, nx_s1y = 0.f, nx_s1z = 0.f;
        auto stage1 = [&](int w_) {
            int g_, t0_, t1_, job_, et_;
            work_item(wk, w_, n_tiles, g_, t0_, t1_);
            locate(pref, n_jobs, g_, job_, et_);
            const ddp_tpconv_edges_t &ed_ = jobs.job[job_].ed;
            nx_ne = min(__ldg(ed_.n_edges_dev), ed_.edge_cap);
            const int e_ = et_ * TILE_M + r;
            if (e_ < ed_.edge_cap) {
                nx_agg = __ldg(ed_.agg + e_);
                nx_gather = __ldg(ed_.gather + e_);
                if (L2) {
                    const float *shp = ed_.sh + (size_t)e_ * 9;       // [s0 | s1 (3) | s2 (5)]: rows are not 16-byte aligned
                    nx_s0 = __ldg(shp); nx_s1x = __ldg(shp + 1); nx_s1y = __ldg(shp + 2); nx_s1z = __ldg(shp + 3);
                } else {
                    const float4 sh4 = __ldg(reinterpret_cast<const float4 *>(ed_.sh + (size_t)e_ * 4));
                    nx_s0 = sh4.x; nx_s1x = sh4.y; nx_s1y = sh4.z; nx_s1z = sh4.w;
                }
            }
        };
        if ((int)blockIdx.x < n_items) stage1(blockIdx.x);
        for (int w = blockIdx.x; w < n_items; w += gridDim.x, ++it) {
            if (tracer && wg == 0) trace_ev(jobs.trace, 2, it * (n_tiles + 1), 0);     // item set-up (free row of the warpgroup-1 trace)
            int g, t0, t1, job, et;
            work_item(wk, w, n_tiles, g, t0, t1);
            const int nt = t1 - t0;
            locate(pref, n_jobs, g, job, et);
            const ddp_tpconv_edges_t &ed = jobs.job[job].ed;
            float *__restrict__ sum = jobs.job[job].sum;
            const int e = et * TILE_M + r;
            const bool valid = e < nx_ne;
            const int ab = it % C::NBUF;
            uint8_t *a_hi = a_base + (size_t)ab * C::A_BYTES * (SPLIT ? 2 : 1);
            uint8_t *a_lo = a_hi + C::A_BYTES;
            if (tracer && wg == 0) trace_ev(jobs.trace, 2, it * (n_tiles + 1), 1);
            const int agg = valid ? nx_agg : 0;
            float inv_deg = 1.f;                         // pre-normalised accumulation: 1 / max(in-degree of agg, 1)
            if (valid && ed.agg_deg != nullptr) inv_deg = __frcp_rn((float)max(__ldg(ed.agg_deg + agg), 1));
            // invalid rows read node 0 and are never written back
            const float *xg = ed.x + (valid ? (size_t)nx_gather * ed.ldx : (size_t)0);
            // every basis row is linear in the edge harmonics: scaling them applies the scatter-mean for free
            const float s0 = valid ? nx_s0 * inv_deg : 0.f, s1x = valid ? nx_s1x * inv_deg : 0.f;
            const float s1y = valid ? nx_s1y * inv_deg : 0.f, s1z = valid ? nx_s1z * inv_deg : 0.f;
            // runs of equal aggregation nodes inside this warp's 32 edges: seg = off | steps << 8 | is_tail << 16
            // (steps = 0: no pre-reduction, e.g. fewer than half of the lanes would merge)
            int seg = 0;
            {
                const int lane_ = r & 31;
                const int key = valid ? agg : -1 - r;
                const int prev = __shfl_up_sync(0xffffffffu, key, 1);
                const unsigned heads = __ballot_sync(0xffffffffu, lane_ == 0 || prev != key);
                const int off = lane_ - (31 - __clz((int)(heads & (0xffffffffu >> (31 - lane_)))));
                const int maxoff = __reduce_max_sync(0xffffffffu, off);
                if (DDP_UMMA_SEGSCAN && __popc(heads) <= 16)
                    seg = off | ((32 - __clz(maxoff)) << 8) | ((lane_ == 31 || ((heads >> (lane_ + 1)) & 1u)) ? 1 << 16 : 0);
            }
            if (tracer && wg == 0) trace_ev(jobs.trace, 2, it * (n_tiles + 1), 2);
            // this warpgroup's tiles of the item: those in its accumulator (acc_of), i.e. every other one from tt_first
            const int tt_first = (int)((wg ^ (uint32_t)nt) & 1u);
            // node features of the first own weight tile (registers; every tile prefetches the next own one's)
            float xn[C::XN];
            uint4 tdw = *reinterpret_cast<const uint4 *>(&tiles[min(t0 + tt_first, n_tiles - 1)]);
            if (tt_first < nt) x_prefetch_tile<NS, NV, C::ROWS_S, C::XN>(xg, tdw, f_in, xn);
            if (tracer && wg == 0) trace_ev(jobs.trace, 2, it * (n_tiles + 1), 3);

            // (the in-degree load and the prefetch are in flight under the conversion)
            if (wg == 0) convert_hidden(a_hi, a_lo, it);
            if (w + (int)gridDim.x < n_items) stage1(w + (int)gridDim.x);

            // ---- weight tiles: TMEM accumulator x tensor-product basis -> per-edge output registers ----
            // Every tile has one basis kind; its node features arrive in registers (prefetched during the previous own
            // tile); the accumulator is read 16 columns at a time with the next tcgen05.ld in flight under the FMAs.
            // Scalar tiles: ROWS_S rows in one pass; vector tiles: up to 2 NV rows in two passes of NV rows.
            // The partial sums of an output block are zeroed at the warpgroup's first tile of the block (or of a split
            // item) and flushed at its last one: when the two interleaved tile sequences are of unequal length both
            // warpgroups hold partial sums of the same block and both add them.
            float acc[NS];
            float u[NV];                                 // x (x) s1 tiles: scalar sums of the current run (see kind 2)
            bool u_live = false;
            int prev_off = -1;
#pragma unroll 1
            for (int tt = tt_first; tt < nt; tt += 2) {
                [[maybe_unused]] const int titer = it * (n_tiles + 1) + 1 + tt;    // trace row (full items)
                const int t = t0 + tt;
                const int kind = (int)((tdw.x >> 16) & 0xffu), n_rows = (int)(tdw.x >> 24);
                const int out_off = (int)(tdw.y & 0xffffu);
                const bool own_next = tt + 2 < nt;
                uint4 tdn = tdw;
                if (own_next) tdn = *reinterpret_cast<const uint4 *>(&tiles[t + 2]);
                const bool blk_first = out_off != prev_off;
                const bool blk_last = !own_next || (int)(tdn.y & 0xffffu) != out_off;
                prev_off = out_off;
                if (blk_first) {
#pragma unroll
                    for (int o = 0; o < NS; ++o) acc[o] = 0.f;
                }
                uint32_t w[2][16];
                if (kind < 2) {
                    float b[C::ROWS_S];
                    if (kind == 0) {
#pragma unroll
                        for (int rr = 0; rr < C::ROWS_S; ++rr) b[rr] = rr < n_rows ? xn[rr] * s0 : 0.f;
                    } else {
#pragma unroll
                        for (int rr = 0; rr < C::ROWS_S; ++rr)
                            b[rr] = rr < n_rows ? xn[3 * rr] * s1x + xn[3 * rr + 1] * s1y + xn[3 * rr + 2] * s1z : 0.f;
                    }
                    if (own_next) x_prefetch_tile<NS, NV, C::ROWS_S, C::XN>(xg, tdn, f_in, xn);
                    if (tracer) trace_ev(jobs.trace, 1 + wg, titer, 0);
                    DDP_WAIT(&tmem_full[wg], tf_phase, 9, it, tt);
                    tf_phase ^= 1u;
                    tc_fence_after();
                    if (tracer) trace_ev(jobs.trace, 1 + wg, titer, 1);
                    tmem_ld16_async(taddr, w[0]);
                    constexpr int NCH = (C::NVAL_S + 15) / 16;
#pragma unroll
                    for (int c16 = 0; c16 < NCH; ++c16) {
                        tmem_wait16(w[c16 & 1]);
                        if (c16 + 1 < NCH) tmem_ld16_async(taddr + (uint32_t)((c16 + 1) * 16), w[(c16 + 1) & 1]);
#pragma unroll
                        for (int q = 0; q < 16; ++q) {
                            const int c = c16 * 16 + q;
                            if (DDP_DIAG_EPI >= 2 && c < C::NVAL_S) acc[c % NS] = fmaf(__uint_as_float(w[c16 & 1][q]), b[c / NS], acc[c % NS]);
                        }
                    }
                    tc_fence_before();
                    mbar_arrive(&tmem_empty[wg]);
                    if (tracer) trace_ev(jobs.trace, 1 + wg, titer, 2);
                    if (blk_last) {
                        if (valid && ed.out_scale != nullptr) {              // block offsets and widths are even: 8-byte loads
                            const float2 *sc2 = reinterpret_cast<const float2 *>(ed.out_scale + out_off);
#pragma unroll
                            for (int o = 0; o < NS; o += 2) {
                                const float2 v = __ldg(sc2 + (o >> 1));
                                acc[o] *= v.x;
                                acc[o + 1] *= v.y;
                            }
                        }
                        const int steps = (seg >> 8) & 0xff;
                        if (steps) seg_scan<NS>(acc, seg & 0xff, steps);
                        if (valid && (steps == 0 || (seg >> 16))) flush_row<NS, FIXED>(sum, (size_t)agg * f_out + out_off, acc, jobs.status);
                    }
                    if (tracer) trace_ev(jobs.trace, 1 + wg, titer, 3);
                } else if (kind == 2) {
                    // x (x) s1 tile (up to 2 NV scalar inputs): out[o][k] += s1[k] * sum_rr w[rr][o] x[rr].  The scalar sums
                    // u[o] are accumulated over the run of such tiles -- one FMA per weight, the basis is the node feature
                    // itself -- and expanded with the edge harmonics when the run ends (next own tile of another kind / block).
                    if (!u_live) {
#pragma unroll
                        for (int o = 0; o < NV; ++o) u[o] = 0.f;
                        u_live = true;
                    }
#pragma unroll
                    for (int rr = 0; rr < C::ROWS_V; ++rr) xn[rr] = rr < n_rows ? xn[rr] : 0.f;     // padding columns are zero, their x is not
                    if (tracer) trace_ev(jobs.trace, 1 + wg, titer, 0);
                    DDP_WAIT(&tmem_full[wg], tf_phase, 10, it, tt);
                    tf_phase ^= 1u;
                    tc_fence_after();
                    if (tracer) trace_ev(jobs.trace, 1 + wg, titer, 1);
                    constexpr int NCOLS = C::ROWS_V * NV, NCH = NCOLS / 16, REM = NCOLS % 16;
                    static_assert(REM == 0 || REM == 8, "x (x) s1 tile remainder is read with one x8 load");
                    tmem_ld16_async(taddr, w[0]);
#pragma unroll
                    for (int c16 = 0; c16 < NCH + (REM ? 1 : 0); ++c16) {
                        tmem_wait16(w[c16 & 1]);
                        if (c16 + 1 < NCH) tmem_ld16_async(taddr + (uint32_t)((c16 + 1) * 16), w[(c16 + 1) & 1]);
                        else if (c16 + 1 == NCH && REM) tmem_ld8_async(taddr + (uint32_t)((c16 + 1) * 16), w[(c16 + 1) & 1]);
                        if (c16 * 16 < n_rows * NV) {            // a short tile's accumulator is stale beyond its own (padded) columns
#pragma unroll
                            for (int q = 0; q < 16; ++q) {
                                const int c = c16 * 16 + q;
                                if (DDP_DIAG_EPI >= 2 && c < NCOLS) u[c % NV] = fmaf(__uint_as_float(w[c16 & 1][q]), xn[c / NV], u[c % NV]);
                            }
                        }
                    }
                    tc_fence_before();
                    mbar_arrive(&tmem_empty[wg]);
                    if (tracer) trace_ev(jobs.trace, 1 + wg, titer, 2);
                    // (the accumulator is free again: everything below overlaps the next MMAs into it)
                    if (own_next) x_prefetch_tile<NS, NV, C::ROWS_S, C::XN>(xg, tdn, f_in, xn);
                    if (blk_last || (int)((tdn.x >> 16) & 0xffu) != 2) {
#pragma unroll
                        for (int o = 0; o < NV; ++o) {
                            acc[3 * o] = fmaf(u[o], s1x, acc[3 * o]);
                            acc[3 * o + 1] = fmaf(u[o], s1y, acc[3 * o + 1]);
                            acc[3 * o + 2] = fmaf(u[o], s1z, acc[3 * o + 2]);
                        }
                        u_live = false;
                    }
                } else {
                    // vector inputs (kinds 3, 4, 5): NV basis rows x NV outputs, three FMAs per weight
                    float bx[NV], by[NV], bz[NV];
                    if (kind == 3) {
#pragma unroll
                        for (int rr = 0; rr < NV; ++rr) {
                            const bool on = rr < n_rows;
                            bx[rr] = on ? xn[3 * rr] * s0 : 0.f; by[rr] = on ? xn[3 * rr + 1] * s0 : 0.f; bz[rr] = on ? xn[3 * rr + 2] * s0 : 0.f;
                        }
                    } else if (L2 && kind == 5) {
                        // b_k = sum_{i,j} C[i][j][k] x_i s2_j: fold the five l = 2 harmonics of the edge into a 3 x 3 matrix
                        // first (45 uniform table reads, 2 such tiles per edge tile), then apply it to every input vector
                        const float *c5 = reinterpret_cast<const float *>(jobs.job[0].image + hdr->ctab5_off) + 45 * (int)((tdw.y >> 24) & 0xffu);
                        float m[3][3] = {{0.f, 0.f, 0.f}, {0.f, 0.f, 0.f}, {0.f, 0.f, 0.f}};
                        if (valid) {
                            const float *s2p = ed.sh + (size_t)e * 9 + 4;
#pragma unroll
                            for (int j = 0; j < 5; ++j) {
                                const float sj = __ldg(s2p + j) * inv_deg;
#pragma unroll
                                for (int i = 0; i < 3; ++i)
#pragma unroll
                                    for (int k = 0; k < 3; ++k) m[i][k] = fmaf(__ldg(c5 + (i * 5 + j) * 3 + k), sj, m[i][k]);
                            }
                        }
#pragma unroll
                        for (int rr = 0; rr < NV; ++rr) {
                            const bool on = rr < n_rows;
                            const float ax = on ? xn[3 * rr] : 0.f, ay = on ? xn[3 * rr + 1] : 0.f, az = on ? xn[3 * rr + 2] : 0.f;
                            bx[rr] = ax * m[0][0] + ay * m[1][0] + az * m[2][0];
                            by[rr] = ax * m[0][1] + ay * m[1][1] + az * m[2][1];
                            bz[rr] = ax * m[0][2] + ay * m[1][2] + az * m[2][2];
                        }
                    } else {
#pragma unroll
                        for (int rr = 0; rr < NV; ++rr) {
                            const bool on = rr < n_rows;
                            const float ax = on ? xn[3 * rr] : 0.f, ay = on ? xn[3 * rr + 1] : 0.f, az = on ? xn[3 * rr + 2] : 0.f;
                            bx[rr] = ay * s1z - az * s1y; by[rr] = az * s1x - ax * s1z; bz[rr] = ax * s1y - ay * s1x;
                        }
                    }
                    // the basis rows are in registers: fetch the next own tile's node features
                    if (own_next) x_prefetch_tile<NS, NV, C::ROWS_S, C::XN>(xg, tdn, f_in, xn);
                    if (tracer) trace_ev(jobs.trace, 1 + wg, titer, 0);
                    DDP_WAIT(&tmem_full[wg], tf_phase, 10, it, tt);
                    tf_phase ^= 1u;
                    tc_fence_after();
                    if (tracer) trace_ev(jobs.trace, 1 + wg, titer, 1);
                    constexpr int NCH = C::PASS_COLS / 16, REM = C::PASS_COLS % 16;
                    static_assert(REM == 0 || REM == 4, "vector tile remainder is read with one x4 load");
                    if (NCH > 0) tmem_ld16_async(taddr, w[0]); else tmem_ld4_async(taddr, w[0]);
#pragma unroll
                    for (int c16 = 0; c16 < NCH + (REM ? 1 : 0); ++c16) {
                        tmem_wait16(w[c16 & 1]);
                        if (c16 + 1 < NCH) tmem_ld16_async(taddr + (uint32_t)((c16 + 1) * 16), w[(c16 + 1) & 1]);
                        else if (c16 + 1 == NCH && REM) tmem_ld4_async(taddr + (uint32_t)((c16 + 1) * 16), w[(c16 + 1) & 1]);
#pragma unroll
                        for (int q = 0; q < 16; ++q) {
                            const int c = c16 * 16 + q;
                            if (c < C::PASS_COLS) {
                                const int rr = c / NV, o = c % NV;
                                const float wv = __uint_as_float(w[c16 & 1][q]);
                                acc[3 * o] = fmaf(wv, bx[rr], acc[3 * o]);
                                acc[3 * o + 1] = fmaf(wv, by[rr], acc[3 * o + 1]);
                                acc[3 * o + 2] = fmaf(wv, bz[rr], acc[3 * o + 2]);
                            }
                        }
                    }
                    tc_fence_before();
                    mbar_arrive(&tmem_empty[wg]);
                    if (tracer) trace_ev(jobs.trace, 1 + wg, titer, 2);
                }
                if (kind >= 2) {
                    if (blk_last) {
                        if (valid && ed.out_scale != nullptr) {
                            const float2 *sc2 = reinterpret_cast<const float2 *>(ed.out_scale + out_off);
#pragma unroll
                            for (int o = 0; o < 3 * NV; o += 2) {
                                const float2 v = __ldg(sc2 + (o >> 1));
                                acc[o] *= v.x;
                                acc[o + 1] *= v.y;
                            }
                        }
                        const int steps = (seg >> 8) & 0xff;
                        if (steps) seg_scan<3 * NV>(acc, seg & 0xff, steps);
                        if (valid && (steps == 0 || (seg >> 16))) flush_row<3 * NV, FIXED>(sum, (size_t)agg * f_out + out_off, acc, jobs.status);
                    }
                    if (tracer) trace_ev(jobs.trace, 1 + wg, titer, 3);
                }
                tdw = tdn;
            }
        }
    }
    // ------------------------------------------------------------------------------------------ teardown
    tc_fence_before();
    __syncthreads();
    if (warp == 5) tmem_dealloc(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------ host: packing
struct HostPlan {
    Header h;
    std::vector<TileDesc> tiles;
    std::vector<std::vector<std::pair<int, float>>> tile_cols;  // per tile: (weight column or -1, scale) per UMMA column
    std::vector<float> ctab5;                                   // 45 floats per kind-5 group
};

static bool pick_cfg(int ns, int nv, int &ks) {
    if (ns == 60 && nv == 10) { ks = 64; return true; }
    if (ns == 24 && nv == 6) { ks = 32; return true; }
    if (ns == 16 && nv == 4) { ks = 32; return true; }
    return false;
}

// Classify a row group of a FasterTensorProduct-shaped spec from its dims and coefficient pattern.
static int group_kind(const ddp_tp_group_t &g, const float *ctab, float &scale) {
    const float *c = ctab + g.c_off;
    if (g.d1 == 1 && g.d2 == 1 && g.d_out == 1) { scale = c[0]; return 0; }
    if (g.d1 == 3 && g.d2 == 3 && g.d_out == 1) { scale = c[0]; return 1; }          // delta_ij * scale
    if (g.d1 == 1 && g.d2 == 3 && g.d_out == 3) { scale = c[0]; return 2; }          // delta_jk * scale
    if (g.d1 == 3 && g.d2 == 1 && g.d_out == 3) { scale = c[0]; return 3; }          // delta_ik * scale
    if (g.d1 == 3 && g.d2 == 3 && g.d_out == 3) { scale = c[(0 * 3 + 1) * 3 + 2]; return 4; }  // eps_ijk * scale
    if (g.d1 == 3 && g.d2 == 5 && g.d_out == 3) { scale = 1.f; return 5; }           // C(1,2,1): the table itself goes into the image
    return -1;
}

static int build_plan(const ddp_tpconv_t &c, const ddp_tp_group_t *groups, const float *ctab_host, int mode, HostPlan &P) {
    int ks;
    const int ns = c.ns;
    // vector multiplicity = mul_out of the first vector-output group
    int nv = 0;
    for (int g = 0; g < c.n_groups; ++g)
        if (groups[g].d_out == 3) { nv = groups[g].mul_out; break; }
    if (nv == 0) nv = (ns == 60) ? 10 : (ns == 24 ? 6 : 4);
    if (!pick_cfg(ns, nv, ks)) return DDP_E_UNSUPPORTED;
    if (c.k1 != 3 * ns || c.hid != 3 * ns || c.n_emb != ns || (c.sh_dim != 4 && c.sh_dim != 9)) return DDP_E_UNSUPPORTED;
    const bool ts = use_ts(mode != 0);
    const int rows_s = rows_scalar(ns, ts), rows_v = rows_vector(nv);
    Header &h = P.h;
    memset(&h, 0, sizeof(h));
    h.magic = MAGIC; h.mode = mode; h.ns = ns; h.nv = nv; h.ks = ks; h.kp = 3 * ks; h.n1 = 3 * ks;
    h.stage_k = stage_k_of(ks, mode != 0); h.f_in = c.f_in; h.f_out = c.f_out; h.sh_dim = c.sh_dim;
    // groups sharing (out_off, d_out) form one weight block (one accumulation of the kernel); they are contiguous in
    // w_off order.  Every tile covers rows of ONE group, so its basis kind and x stride are uniform.
    int g = 0;
    while (g < c.n_groups) {
        int g_end = g;
        while (g_end < c.n_groups && groups[g_end].out_off == groups[g].out_off && groups[g_end].d_out == groups[g].d_out) ++g_end;
        const bool vec = groups[g].d_out == 3;
        const int mul_out = groups[g].mul_out;
        if (mul_out != (vec ? nv : ns)) return DDP_E_UNSUPPORTED;
        const size_t first_tile = P.tiles.size();
        for (int q = g; q < g_end; ++q) {
            float sc;
            const int kind = group_kind(groups[q], ctab_host, sc);
            if (kind < 0 || (vec != (kind >= 2))) return DDP_E_UNSUPPORTED;
            if (kind == 5 && c.sh_dim != 9) return DDP_E_UNSUPPORTED;
            if (groups[q].sh_off != (kind == 5 ? 4 : ((kind == 0 || kind == 3) ? 0 : 1))) return DDP_E_UNSUPPORTED;
            int table5 = 0;
            if (kind == 5) {
                table5 = (int)P.ctab5.size() / 45;
                if (table5 > 255) return DDP_E_UNSUPPORTED;
                P.ctab5.insert(P.ctab5.end(), ctab_host + groups[q].c_off, ctab_host + groups[q].c_off + 45);
            }
            const int d1 = groups[q].d1;
            // rows per tile: scalar tiles ROWS_S; x (x) s1 tiles 2 NV (two epilogue passes); stride-3 vector kinds NV
            const int per = !vec ? rows_s : (kind == 2 ? rows_v : nv);
            for (int r0 = 0; r0 < groups[q].mul_in; r0 += per) {
                const int nr = std::min(per, groups[q].mul_in - r0);
                TileDesc td;
                memset(&td, 0, sizeof(td));
                td.n_cols = (uint16_t)(vec ? ncol_vector(nv, nr) : ncol_scalar(ns, ts));
                td.kind = (uint8_t)kind;
                td.ctab5 = (uint8_t)table5;
                td.n_rows = (uint8_t)nr;
                td.out_off = (uint16_t)groups[g].out_off;
                const int xo = groups[q].x_off + r0 * d1;   // first gathered feature the tile reads
                td.x_off = (uint16_t)xo;
                std::vector<std::pair<int, float>> cols(td.n_cols, {-1, 0.f});
                for (int rr = 0; rr < nr; ++rr)
                    for (int o = 0; o < mul_out; ++o) cols[rr * mul_out + o] = {groups[q].w_off + (r0 + rr) * mul_out + o, sc};
                P.tiles.push_back(td);
                P.tile_cols.push_back(cols);
            }
        }
        if (P.tiles.size() == first_tile) return DDP_E_UNSUPPORTED;
        P.tiles[first_tile].flags |= 1;
        P.tiles.back().flags |= 4;
        g = g_end;
    }
    // Tile order = consumption order.  The two epilogue warpgroups take alternate tiles (one per TMEM accumulator), so the
    // tiles of the leading blocks (sequence A, about half of the MMA cost) are interleaved with those of the remaining blocks
    // (sequence B): each warpgroup then owns whole output blocks -- one flush per block, as with a single warpgroup -- and
    // the vector tiles of one sequence (slow epilogue) pair with scalar tiles of the other where the layer is symmetric.
    // Left-over tiles of the longer sequence alternate between the warpgroups, which then both flush partial sums.
    {
        const int n = (int)P.tiles.size();
        long total = 0, cum = 0, best_d = 0;
        for (const TileDesc &td : P.tiles) total += td.n_cols;
        int cut = n;
        for (int t = 0; t < n; ++t) {
            const long d = labs(2 * cum - total);
            if (t > 0 && (P.tiles[t].flags & 1) && (cut == n || d < best_d)) { cut = t; best_d = d; }
            cum += P.tiles[t].n_cols;
        }
        if (cut < n) {
            std::vector<TileDesc> tiles;
            std::vector<std::vector<std::pair<int, float>>> cols;
            for (int i = 0, j = cut; i < cut || j < n;) {
                if (i < cut) { tiles.push_back(P.tiles[i]); cols.push_back(std::move(P.tile_cols[i])); ++i; }
                if (j < n) { tiles.push_back(P.tiles[j]); cols.push_back(std::move(P.tile_cols[j])); ++j; }
            }
            P.tiles.swap(tiles);
            P.tile_cols.swap(cols);
            // flags 1 / 4: first / last tile of its block in the new order (informative: the kernel compares block offsets)
            for (int t = 0; t < n; ++t) {
                bool first = true, last = true;
                for (int u = 0; u < t; ++u) first = first && P.tiles[u].out_off != P.tiles[t].out_off;
                for (int u = t + 1; u < n; ++u) last = last && P.tiles[u].out_off != P.tiles[t].out_off;
                P.tiles[t].flags = (uint8_t)((P.tiles[t].flags & ~5) | (first ? 1 : 0) | (last ? 4 : 0));
            }
        }
    }
    h.n_tiles = (int)P.tiles.size();
    if (h.n_tiles > 64) return DDP_E_UNSUPPORTED;
    int64_t off = (sizeof(Header) + 127) / 128 * 128;
    h.tiles_off = off;
    off += (int64_t)((h.n_tiles * sizeof(TileDesc) + 127) / 128 * 128);
    h.n_ctab5 = (int)P.ctab5.size() / 45;
    h.ctab5_off = off;
    off += (int64_t)((P.ctab5.size() * sizeof(float) + 127) / 128 * 128);
    h.slabs_off = off;
    int64_t slab_total = (int64_t)slab_bytes(h.n1, h.stage_k, mode) * (h.kp / h.stage_k);
    for (auto &td : P.tiles) slab_total += (int64_t)slab_bytes(td.n_cols, h.stage_k, mode) * (h.kp / h.stage_k);
    h.total_bytes = off + slab_total;
    h.n_slabs_per_edge_tile = (h.n_tiles + 1) * (h.kp / h.stage_k);
    return 0;
}

static inline uint16_t f2bf(float f) {
    uint32_t u;
    memcpy(&u, &f, 4);
    if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40);
    u += 0x7fffu + ((u >> 16) & 1u);
    return (uint16_t)(u >> 16);
}
static inline float bf2f(uint16_t b) {
    uint32_t u = (uint32_t)b << 16;
    float f;
    memcpy(&f, &u, 4);
    return f;
}

// Write one [n_cols x KP] operand (value(n, k) callback) as K-slabs in UMMA no-swizzle core-matrix order:
// slab ks: [k-chunk (stage_k/8)][row group (n_cols/8)][8 rows][8 elements]; split mode appends the lo image.
template <class F>
static uint8_t *emit_operand(uint8_t *dst, int n_cols, int kp, int stage_k, int mode, F value) {
    for (int ks = 0; ks < kp / stage_k; ++ks) {
        uint16_t *hi = reinterpret_cast<uint16_t *>(dst);
        uint16_t *lo = hi + (size_t)n_cols * stage_k;
        for (int kc = 0; kc < stage_k / 8; ++kc)
            for (int n = 0; n < n_cols; ++n)
                for (int q = 0; q < 8; ++q) {
                    const float v = value(n, ks * stage_k + kc * 8 + q);
                    const size_t idx = ((size_t)kc * (n_cols / 8) + n / 8) * 64 + (n % 8) * 8 + q;
                    const uint16_t h = f2bf(v);
                    hi[idx] = h;
                    if (mode) lo[idx] = f2bf(v - bf2f(h));
                }
        dst += slab_bytes(n_cols, stage_k, mode);
    }
    return dst;
}

}  // namespace umma

extern "C" int64_t ddp_tpconv_pack(const ddp_tpconv_t *conv, const ddp_tp_group_t *groups_host, const float *ctab_host,
                                    const float *w1, const float *b1, const float *w2, const float *b2, int32_t mode,
                                    void *packed_host) {
    using namespace umma;
    if (!conv || !groups_host || !ctab_host) return DDP_E_ARG;
    if (mode != 0 && mode != 1) return DDP_E_ARG;
    HostPlan P;
    const int rc = build_plan(*conv, groups_host, ctab_host, mode, P);
    if (rc != 0) return rc;
    if (packed_host == nullptr) return P.h.total_bytes;
    if (!w1 || !b1 || !w2 || !b2) return DDP_E_ARG;
    const Header &h = P.h;
    uint8_t *base = static_cast<uint8_t *>(packed_host);
    memset(base, 0, (size_t)h.total_bytes);
    memcpy(base, &h, sizeof(h));
    memcpy(base + h.tiles_off, P.tiles.data(), P.tiles.size() * sizeof(TileDesc));
    if (!P.ctab5.empty()) memcpy(base + h.ctab5_off, P.ctab5.data(), P.ctab5.size() * sizeof(float));
    const int ns = h.ns, ks = h.ks, hid = conv->hid, k1 = conv->k1;
    uint8_t *dst = base + h.slabs_off;
    // GEMM1 operand: rows n = hidden unit, k' = source * ks + j; bias in (source 0, j = ns); row `hid` regenerates the one
    dst = emit_operand(dst, h.n1, h.kp, h.stage_k, mode, [&](int n, int kq) -> float {
        const int s = kq / ks, j = kq % ks;
        if (n < hid) {
            if (j < ns) return w1[(size_t)n * k1 + s * ns + j];
            if (s == 0 && j == ns) return b1[n];
            return 0.f;
        }
        return (n == hid && s == 0 && j == ns) ? 1.f : 0.f;
    });
    // GEMM2 operands: rows = UMMA columns of the tile, k = hidden unit (bias at k = hid)
    for (size_t t = 0; t < P.tiles.size(); ++t) {
        const auto &cols = P.tile_cols[t];
        dst = emit_operand(dst, P.tiles[t].n_cols, h.kp, h.stage_k, mode, [&](int n, int k) -> float {
            const int wc = cols[n].first;
            if (wc < 0) return 0.f;
            if (k < hid) return cols[n].second * w2[(size_t)wc * hid + k];
            if (k == hid) return cols[n].second * b2[wc];
            return 0.f;
        });
    }
    return (dst - base) == h.total_bytes ? 0 : DDP_E_SHAPE;
}

template <int NS, int NV, int KS, bool SPLIT, bool L2, bool FIXED>
static int launch_umma_l(const umma::Jobs &jobs, int tiles_cap, cudaStream_t st) {
    using C = umma::Cfg<NS, NV, KS, SPLIT>;
    auto kern = umma::tpconv_umma_kernel<NS, NV, KS, SPLIT, L2, FIXED>;
    static bool configured[DDP_MAX_DEVICES] = {false};
    cudaError_t err = ddp_smem_opt_in(kern, C::SMEM, configured);
    if (err != cudaSuccess) return (int)err;
    const int grid = tiles_cap < ddp_num_sms() ? tiles_cap : ddp_num_sms();
    kern<<<grid, umma::N_THREADS, C::SMEM, st>>>(jobs);
    DDP_LAUNCH_CHECK();
    return 0;
}

template <int NS, int NV, int KS, bool SPLIT, bool FIXED>
static int launch_umma(const umma::Jobs &jobs, int tiles_cap, cudaStream_t st, bool l2) {
    return l2 ? launch_umma_l<NS, NV, KS, SPLIT, true, FIXED>(jobs, tiles_cap, st) : launch_umma_l<NS, NV, KS, SPLIT, false, FIXED>(jobs, tiles_cap, st);
}

static long long *g_umma_trace = nullptr;
extern "C" int ddp_tpconv_umma_set_trace(void *trace_dev) {
#ifdef DDP_UMMA_TRACE
    g_umma_trace = static_cast<long long *>(trace_dev);
    return 3 * umma::TRACE_TILES * umma::TRACE_EVENTS;      // int64 slots the buffer must hold (watchdog build: 148 x 12 x 4 of them)
#else
    (void)trace_dev;
    return DDP_E_UNSUPPORTED;                               // library built without -DDDP_UMMA_TRACE
#endif
}

template <bool FIXED>
static int tpconv_umma_group(const ddp_tpconv_t *const *convs, const void *const *packed, int32_t mode, const ddp_tpconv_edges_t *const *edges,
                             float *const *sums, int32_t n_jobs, uint32_t *status, void *stream) {
    if (!convs || !packed || !edges || !sums || (FIXED && !status)) return DDP_E_ARG;
    if (n_jobs <= 0) return 0;
    if (n_jobs > umma::MAX_JOBS) return DDP_E_SHAPE;
    umma::Jobs jobs;
    memset(&jobs, 0, sizeof(jobs));
    const ddp_tpconv_t &c0 = *convs[0];
    jobs.f_in = c0.f_in;
    jobs.f_out = c0.f_out;
    jobs.trace = g_umma_trace;
    jobs.status = status;
    int tiles_cap = 0;
    for (int j = 0; j < n_jobs; ++j) {
        if (!convs[j] || !packed[j] || !edges[j] || !sums[j]) return DDP_E_ARG;
        const ddp_tpconv_t &c = *convs[j];
        const ddp_tpconv_edges_t &e = *edges[j];
        // one tile table for the whole launch: same irreps / weight layout in every job
        if (c.ns != c0.ns || c.f_in != c0.f_in || c.f_out != c0.f_out || c.w_numel != c0.w_numel || c.n_groups != c0.n_groups ||
            c.sh_dim != c0.sh_dim)
            return DDP_E_SHAPE;
        if (c.sh_dim != 4 && c.sh_dim != 9) return DDP_E_UNSUPPORTED;
        if (!e.emb || !e.x || !e.gather || !e.sh || !e.agg || !e.n_edges_dev || !e.p1 || !e.p2 || !e.i1 || !e.i2) return DDP_E_ARG;
        if (e.ew != nullptr) return DDP_E_UNSUPPORTED;
        if ((e.ldx & 1) || (c.f_out & 1)) return DDP_E_UNSUPPORTED;      // 8-byte aligned rows (vector loads / reductions)
        if (e.edge_cap <= 0) continue;
        umma::Job &jb = jobs.job[jobs.n++];
        jb.image = static_cast<const uint8_t *>(packed[j]);
        jb.ed = e;
        jb.sum = sums[j];
        tiles_cap += (e.edge_cap + umma::TILE_M - 1) / umma::TILE_M;
    }
    if (jobs.n == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    const bool l2 = c0.sh_dim == 9;
    if (c0.ns == 60) return mode ? launch_umma<60, 10, 64, true, FIXED>(jobs, tiles_cap, st, l2) : launch_umma<60, 10, 64, false, FIXED>(jobs, tiles_cap, st, l2);
    if (c0.ns == 24) return mode ? launch_umma<24, 6, 32, true, FIXED>(jobs, tiles_cap, st, l2) : launch_umma<24, 6, 32, false, FIXED>(jobs, tiles_cap, st, l2);
    if (c0.ns == 16) return mode ? launch_umma<16, 4, 32, true, FIXED>(jobs, tiles_cap, st, l2) : launch_umma<16, 4, 32, false, FIXED>(jobs, tiles_cap, st, l2);
    return DDP_E_UNSUPPORTED;
}

extern "C" int ddp_tpconv_umma_group(const ddp_tpconv_t *const *convs, const void *const *packed, int32_t mode,
                                     const ddp_tpconv_edges_t *const *edges, float *const *sums, int32_t n_jobs, void *stream) {
    return tpconv_umma_group<false>(convs, packed, mode, edges, sums, n_jobs, nullptr, stream);
}

extern "C" int ddp_tpconv_umma(const ddp_tpconv_t *conv, const void *packed, int32_t mode, const ddp_tpconv_edges_t *edges,
                               float *sum, void *stream) {
    if (!conv || !packed || !edges || !sum) return DDP_E_ARG;
    return ddp_tpconv_umma_group(&conv, &packed, mode, &edges, &sum, 1, stream);
}

extern "C" int ddp_tpconv_umma_group_fixed(const ddp_tpconv_t *const *convs, const void *const *packed, int32_t mode,
                                           const ddp_tpconv_edges_t *const *edges, int64_t *const *sums, int32_t n_jobs,
                                           uint32_t *status, void *stream) {
    return tpconv_umma_group<true>(convs, packed, mode, edges, reinterpret_cast<float *const *>(sums), n_jobs, status, stream);
}

extern "C" int ddp_tpconv_umma_fixed(const ddp_tpconv_t *conv, const void *packed, int32_t mode, const ddp_tpconv_edges_t *edges,
                                     int64_t *sum, uint32_t *status, void *stream) {
    if (!conv || !packed || !edges || !sum) return DDP_E_ARG;
    return ddp_tpconv_umma_group_fixed(&conv, &packed, mode, &edges, &sum, 1, status, stream);
}
