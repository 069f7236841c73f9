// K1 / K5 on the 5th-generation tensor cores: fp32-accurate GEMM by 3xTF32 error compensation.
//
//   C[M,N] (+)= A[M,K] * B[K,N],   A = A_hi + A_lo,  B = B_hi + B_lo  (hi = top 19 bits, lo = remainder)
//   C ~= A_hi*B_hi + A_lo*B_hi + A_hi*B_lo        (fp32 accumulation in TMEM; dropped term ~2^-20)
//
// Structure (one persistent CTA per SM, 320 threads, warp-specialised):
//   warp 0      TMA producer: cp.async.bulk.tensor tiles of A (raw fp32) and of the pre-split, pre-transposed
//               weights B_hi / B_lo ([N,K], K-major) into a 128B-swizzled shared-memory ring
//   warps 2-5   splitter: rewrite the raw A tile in place as A_hi and write A_lo beside it
//   warp 1      MMA issuer: one thread issues tcgen05.mma.kind::tf32 (M=128, N=BN, K=8) x3 per K-step,
//               accumulators in TMEM (two 256-column buffers, ping-pong across tiles)
//   warps 6-9   epilogue: tcgen05.ld accumulator rows -> registers -> global (optional C += )
// mbarriers: full (TMA->splitter/MMA), conv (splitter->MMA), empty (MMA commit->TMA),
//            tfull (MMA commit->epilogue), tempty (epilogue->MMA).
// The projection GEMMs this serves are the re-associated `a.mm(edge_h)` of GAT/layers.py:137
// (SURVEY.md 8 a-4) and its autograd products; weights are tiny so B is split once per call on the device.
#include <cuda.h>
#include <stdlib.h>
#include "spk_common.cuh"
#include "spk_gemm.cuh"

namespace spk {
namespace {

constexpr int TC_BM = 128;
constexpr int TC_BK = 32;                       // 32 fp32 = 128 B = one swizzle row
constexpr int TC_A_TILE = TC_BM * TC_BK * 4;    // 16 KB
constexpr int TC_THREADS = 320;
constexpr int TC_MAX_STAGES = 4;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred P1;\n\t"
        "LAB_WAIT:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
        "@P1 bra DONE;\n\t"
        "bra LAB_WAIT;\n\t"
        "DONE:\n\t"
        "}" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(tm), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
// multicast form: the box lands at the same CTA-relative offset, and completes on the same CTA-relative mbarrier, in every
// CTA of the cluster named in `mask`
__device__ __forceinline__ void tma_load_2d_mc(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, uint16_t mask) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(dst), "l"(tm), "r"(bar), "r"(c0), "r"(c1), "h"(mask) : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// commit that arrives on the same CTA-relative mbarrier of every CTA in `mask` (frees a multicast-filled stage cluster-wide)
__device__ __forceinline__ void tc_commit_mc(uint32_t bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(bar), "h"(mask) : "memory");
}
__device__ __forceinline__ void tc_mma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum) : "memory");
}
// K-major, 128B-swizzled operand tile: rows of 128 B, 8-row groups 1024 B apart (cute::UMMA::SmemDescriptor)
__device__ __forceinline__ uint64_t make_kmajor_sw128_desc(uint32_t saddr) {
    const uint32_t lo = ((saddr >> 4) & 0x3fffu) | (1u << 16);          // start address | LBO (unused with swizzle)
    const uint32_t hi = (1024u >> 4) | (1u << 14) | (2u << 29);        // SBO | descriptor version 1 | SWIZZLE_128B
    return ((uint64_t)hi << 32) | lo;
}

struct TcParams {
    float* C; long ldc; long M; int N; int K; int BN; int n_tiles_n; int stages; int accumulate; int c_vec;
    int act;                                    // epilogue on the final value: 0 = none, 1 = ELU (GAT/layers.py:175),
                                                // 2 = tanh (GAT_sep_space/models.py:316-320)
    int c_tma;                                  // epilogue stores through shared memory + TMA (coalesced 128 B rows)
    int raw_hi;                                 // the MMA reads the raw fp32 tile as "hi" (kind::tf32 ignores the low 13 mantissa bits)
    int cs;                                     // cluster size (1 or 2): the CTAs of a cluster work on consecutive M tiles of the
                                                // same N tile in lock-step and share every weight tile by TMA multicast
    const int* tile_group;                      // grouped kernel only: group of every 128-row M tile; the weight rows of group g
    const int* n_mtiles;                        // start at row g * N of the stacked B_hi / B_lo; *n_mtiles = M tiles to run
};

// ELU(x) = x (x > 0) else expm1(x); same evaluation as the edge kernels (degree-5 polynomial near 0)
__device__ __forceinline__ float tc_elu(float x) {
    const float big = exp2f(x * 1.4426950408889634f) - 1.0f;
    const float small = x * (1.0f + x * (0.5f + x * (0.16666667f + x * (0.041666668f + x * 0.0083333338f))));
    const float neg = x > -0.125f ? small : big;
    return x > 0.f ? x : neg;
}

// The epilogue activation of act != 0 (the TMA-store epilogues branch once per chunk instead); tanh is the libdevice tanhf
// of tanh_fwd_kernel (spk_convkb.cu, no fast-math), so act = 2 gives the same bits as the product followed by spk_tanh_fwd.
__device__ __forceinline__ float tc_act(float x, int act) { return act == 2 ? tanhf(x) : tc_elu(x); }

// GROUPED: C_g = A_g . B_g for row groups padded to whole M tiles (spk_ent2rel_*): the tile count and each tile's group are
// read from the device, so the launch needs no host-side knowledge of the grouping (cs == 1 only)
template <bool GROUPED>
__global__ void __launch_bounds__(TC_THREADS, 1)
gemm_nn_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmBhi,
                  const __grid_constant__ CUtensorMap tmBlo, const __grid_constant__ CUtensorMap tmC, const TcParams p) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bars[3 * TC_MAX_STAGES + 4];
    __shared__ uint32_t tmem_slot;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t b_tile = (uint32_t)p.BN * 128u;
    const uint32_t stage_bytes = 2u * TC_A_TILE + 2u * b_tile;
    auto a_hi = [&](int s) { return base + (uint32_t)s * stage_bytes; };
    auto a_lo = [&](int s) { return base + (uint32_t)s * stage_bytes + TC_A_TILE; };
    auto b_hi = [&](int s) { return base + (uint32_t)s * stage_bytes + 2u * TC_A_TILE; };
    auto b_lo = [&](int s) { return base + (uint32_t)s * stage_bytes + 2u * TC_A_TILE + b_tile; };
    const uint32_t bar0 = smem_u32(bars);
    auto full = [&](int s) { return bar0 + 8u * s; };
    auto conv = [&](int s) { return bar0 + 8u * (TC_MAX_STAGES + s); };
    auto empty = [&](int s) { return bar0 + 8u * (2 * TC_MAX_STAGES + s); };
    auto tfull = [&](int a) { return bar0 + 8u * (3 * TC_MAX_STAGES + a); };
    auto tempty = [&](int a) { return bar0 + 8u * (3 * TC_MAX_STAGES + 2 + a); };

    const int num_kb = (p.K + TC_BK - 1) / TC_BK;
    const long m_tiles = (p.M + TC_BM - 1) / TC_BM;
    // Work items are "super tiles": cs consecutive M tiles x one N tile, one per cluster and iteration; the CTA of cluster
    // rank r takes M tile (super * cs + r) (possibly past the end: its loads are zero-filled and its stores clipped), so all
    // CTAs of a cluster run the same number of pipeline steps and can share the weight tiles.
    const int cs = p.cs;
    const uint32_t crank = cs > 1 ? cluster_ctarank() : 0u;
    const uint16_t cmask = (uint16_t)((1u << cs) - 1u);
    const long total = GROUPED ? (long)*p.n_mtiles * p.n_tiles_n : ((m_tiles + cs - 1) / cs) * p.n_tiles_n;
    const long first = blockIdx.x / cs, stride = gridDim.x / cs;
    const uint32_t b_slice = b_tile / (uint32_t)cs;               // bytes of this CTA's share of a weight tile
    const int b_rows = p.BN / cs;

    if (threadIdx.x == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmBhi) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmBlo) : "memory");
        for (int s = 0; s < TC_MAX_STAGES; ++s) { mbar_init(full(s), 1); mbar_init(conv(s), 128); mbar_init(empty(s), (uint32_t)cs); }
        for (int a = 0; a < 2; ++a) { mbar_init(tfull(a), 1); mbar_init(tempty(a), 4); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    if (cs > 1) cluster_sync_all();                                // peers' barriers are initialised before anything arrives
    tc_fence_after();
    const uint32_t tmem_base = tmem_slot;

    if (warp == 0) {
        if (lane == 0) {                                           // ---- TMA producer
            uint32_t it = 0;
            for (long tile = first; tile < total; tile += stride) {
                const int m0 = (int)((tile / p.n_tiles_n) * cs + crank) * TC_BM;
                const int n0 = (int)(tile % p.n_tiles_n) * p.BN + (GROUPED ? p.tile_group[tile / p.n_tiles_n] * p.N : 0);
                for (int kb = 0; kb < num_kb; ++kb, ++it) {
                    const int s = it % p.stages;
                    const uint32_t ph = (it / p.stages) & 1u;
                    mbar_wait(empty(s), ph ^ 1u);                   // every CTA of the cluster has released this stage
                    mbar_arrive_expect_tx(full(s), TC_A_TILE + 2u * b_tile);
                    tma_load_2d(a_hi(s), &tmA, full(s), kb * TC_BK, m0);
                    if (cs == 1) {
                        tma_load_2d(b_hi(s), &tmBhi, full(s), kb * TC_BK, n0);
                        tma_load_2d(b_lo(s), &tmBlo, full(s), kb * TC_BK, n0);
                    } else {                                        // my 1/cs of the weight tile, delivered to all CTAs
                        tma_load_2d_mc(b_hi(s) + crank * b_slice, &tmBhi, full(s), kb * TC_BK, n0 + (int)crank * b_rows, cmask);
                        tma_load_2d_mc(b_lo(s) + crank * b_slice, &tmBlo, full(s), kb * TC_BK, n0 + (int)crank * b_rows, cmask);
                    }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {                                           // ---- MMA issuer
            const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(p.BN >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
            uint32_t it = 0, tl = 0;
            for (long tile = first; tile < total; tile += stride, ++tl) {
                const uint32_t acc = tl & 1u, aph = (tl >> 1) & 1u;
                mbar_wait(tempty(acc), aph ^ 1u);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * 256u;
                for (int kb = 0; kb < num_kb; ++kb, ++it) {
                    const int s = it % p.stages;
                    const uint32_t ph = (it / p.stages) & 1u;
                    mbar_wait(full(s), ph);
                    mbar_wait(conv(s), ph);
                    tc_fence_after();
                    const uint64_t dah = make_kmajor_sw128_desc(a_hi(s)), dal = make_kmajor_sw128_desc(a_lo(s));
                    const uint64_t dbh = make_kmajor_sw128_desc(b_hi(s)), dbl = make_kmajor_sw128_desc(b_lo(s));
#pragma unroll
                    for (int ks = 0; ks < TC_BK / 8; ++ks) {
                        if (kb * TC_BK + ks * 8 >= p.K) break;
                        const uint64_t o = (uint64_t)(2 * ks);      // 32 B per K-step, in 16-byte units
                        tc_mma_tf32(d_tmem, dal + o, dbh + o, idesc, (kb | ks) != 0);
                        tc_mma_tf32(d_tmem, dah + o, dbl + o, idesc, 1u);
                        tc_mma_tf32(d_tmem, dah + o, dbh + o, idesc, 1u);
                    }
                    if (cs == 1) tc_commit(empty(s));               // frees the smem stage when these MMAs retire
                    else tc_commit_mc(empty(s), cmask);             // ... in every CTA of the cluster (their copies refill it)
                }
                tc_commit(tfull(acc));                              // accumulator complete -> epilogue
            }
        }
    } else if (warp < 6) {                                         // ---- splitter: raw fp32 -> (hi, lo)
        const int t = threadIdx.x - 64;
        uint32_t it = 0;
        for (long tile = first; tile < total; tile += stride) {
            for (int kb = 0; kb < num_kb; ++kb, ++it) {
                const int s = it % p.stages;
                const uint32_t ph = (it / p.stages) & 1u;
                mbar_wait(full(s), ph);
                const uint32_t hi0 = a_hi(s), lo0 = a_lo(s);
#pragma unroll
                for (int i = 0; i < TC_A_TILE / 16 / 128; ++i) {
                    const uint32_t off = (uint32_t)(t + 128 * i) * 16u;
                    float4 x;
                    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(x.x), "=f"(x.y), "=f"(x.z), "=f"(x.w) : "r"(hi0 + off));
                    float4 h, l;
                    h.x = __uint_as_float(__float_as_uint(x.x) & 0xffffe000u); l.x = x.x - h.x;
                    h.y = __uint_as_float(__float_as_uint(x.y) & 0xffffe000u); l.y = x.y - h.y;
                    h.z = __uint_as_float(__float_as_uint(x.z) & 0xffffe000u); l.z = x.z - h.z;
                    h.w = __uint_as_float(__float_as_uint(x.w) & 0xffffe000u); l.w = x.w - h.w;
                    if (!p.raw_hi)
                        asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(hi0 + off), "f"(h.x), "f"(h.y), "f"(h.z), "f"(h.w) : "memory");
                    asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(lo0 + off), "f"(l.x), "f"(l.y), "f"(l.z), "f"(l.w) : "memory");
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic writes -> visible to the MMA's async proxy
                mbar_arrive(conv(s));
            }
        }
    } else if (p.c_tma) {                                          // ---- epilogue (warps 6..9), coalesced
        // Each warp owns the 32 accumulator rows of its TMEM lane quarter. A 32-column chunk is read with one
        // tcgen05.ld (a lane = one row), written to a 128B-swizzled [32 x 32] staging tile in shared memory and
        // stored (or reduce-added, for C +=) by TMA: full 128 B row segments, clipped at the M / N edges.
        const int q = warp & 3;
        const uint32_t stg0 = base + (uint32_t)p.stages * stage_bytes + (uint32_t)q * 8192u;
        uint32_t tl = 0, sb = 0;
        for (long tile = first; tile < total; tile += stride, ++tl) {
            const uint32_t acc = tl & 1u, aph = (tl >> 1) & 1u;
            const int row0 = (int)((tile / p.n_tiles_n) * cs + crank) * TC_BM + q * 32;
            const int n0 = (int)(tile % p.n_tiles_n) * p.BN;
            mbar_wait(tfull(acc), aph);
            tc_fence_after();
            // A warp whose 32 rows lie past the last row of C has nothing to store, and it must not touch its staging buffers:
            // it commits no bulk group, so `wait_group.read 1` would keep admitting the LAST store of the previous tile as
            // the one allowed reader while its buffer is rewritten with this tile's zeros (lost C += rows; found by
            // test_gemm_nn[20000-52-416]: M tiles 156 = 2 x 148 CTAs + partial last tile).
            for (int c0 = 0; c0 < p.BN && row0 < p.M; c0 += 32) {
                if (n0 + c0 >= p.N) break;
                uint32_t r[32];
                const uint32_t taddr = tmem_base + acc * 256u + (uint32_t)c0 + ((uint32_t)(q * 32) << 16);
                asm volatile(
                    "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
                    "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
                    : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                      "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
                      "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
                      "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                    : "r"(taddr));
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if (p.act == 2) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) r[j] = __float_as_uint(tanhf(__uint_as_float(r[j])));
                } else if (p.act) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) r[j] = __float_as_uint(tc_elu(__uint_as_float(r[j])));
                }
                // the store issued two chunks ago read this staging buffer: wait until at most one store is still reading
                if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
                __syncwarp();
                const uint32_t stg = stg0 + sb * 4096u;
                const uint32_t rowaddr = stg + (uint32_t)lane * 128u;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const uint32_t a = rowaddr + (uint32_t)((j ^ (lane & 7)) << 4);
                    asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(a), "r"(r[4 * j]), "r"(r[4 * j + 1]),
                                 "r"(r[4 * j + 2]), "r"(r[4 * j + 3]) : "memory");
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncwarp();
                if (lane == 0 && row0 < p.M) {                      // (a padding tile past the last row stores nothing)
                    if (p.accumulate)
                        asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%1, %2}], [%3];"
                                     ::"l"(&tmC), "r"(n0 + c0), "r"(row0), "r"(stg) : "memory");
                    else
                        asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group [%0, {%1, %2}], [%3];"
                                     ::"l"(&tmC), "r"(n0 + c0), "r"(row0), "r"(stg) : "memory");
                    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                }
                sb ^= 1u;
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty(acc));
        }
        if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    } else {                                                       // ---- epilogue (warps 6..9), per-thread rows (unaligned C)
        const int q = warp & 3;                                    // TMEM lane quarter this warp may access
        uint32_t tl = 0;
        for (long tile = first; tile < total; tile += stride, ++tl) {
            const uint32_t acc = tl & 1u, aph = (tl >> 1) & 1u;
            const long row = ((tile / p.n_tiles_n) * cs + crank) * TC_BM + q * 32 + lane;
            const int n0 = (int)(tile % p.n_tiles_n) * p.BN;
            mbar_wait(tfull(acc), aph);
            tc_fence_after();
            for (int c0 = 0; c0 < p.BN; c0 += 16) {
                uint32_t r[16];
                const uint32_t taddr = tmem_base + acc * 256u + (uint32_t)c0 + ((uint32_t)(q * 32) << 16);
                asm volatile(
                    "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                    : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                      "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                    : "r"(taddr));
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if (row < p.M) {
                    float* crow = p.C + row * p.ldc;
#pragma unroll
                    for (int j = 0; j < 16; j += 4) {
                        const int col = n0 + c0 + j;
                        if (col >= p.N) break;
                        float4 o = make_float4(__uint_as_float(r[j]), __uint_as_float(r[j + 1]), __uint_as_float(r[j + 2]), __uint_as_float(r[j + 3]));
                        if (p.c_vec && col + 3 < p.N) {
                            if (p.accumulate) o = f4add(o, *reinterpret_cast<const float4*>(crow + col));
                            if (p.act) o = make_float4(tc_act(o.x, p.act), tc_act(o.y, p.act), tc_act(o.z, p.act), tc_act(o.w, p.act));
                            *reinterpret_cast<float4*>(crow + col) = o;
                        } else {
                            const float ov[4] = {o.x, o.y, o.z, o.w};
#pragma unroll
                            for (int k = 0; k < 4; ++k)
                                if (col + k < p.N) {
                                    const float r1 = p.accumulate ? crow[col + k] + ov[k] : ov[k];
                                    crow[col + k] = p.act ? tc_act(r1, p.act) : r1;
                                }
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty(acc));
        }
    }
    tc_fence_before();
    __syncthreads();
    if (cs > 1) cluster_sync_all();                                // no CTA leaves while a peer may still signal its barriers
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}


// ---- 2-CTA (cta_group::2) helpers --------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) {      // acquire at cluster scope
    asm volatile(
        "{\n\t"
        ".reg .pred P1;\n\t"
        "LAB_WAITC:\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 P1, [%0], %1;\n\t"
        "@P1 bra DONEC;\n\t"
        "bra LAB_WAITC;\n\t"
        "DONEC:\n\t"
        "}" ::"r"(bar), "r"(parity) : "memory");
}
// arrive (release at cluster scope) on the mbarrier at the same CTA-relative address in the CTA of cluster rank `rank`
__device__ __forceinline__ void mbar_arrive_remote(uint32_t bar, uint32_t rank) {
    asm volatile(
        "{\n\t"
        ".reg .b32 ra;\n\t"
        "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
        "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n\t"
        "}" ::"r"(bar), "r"(rank) : "memory");
}
__device__ __forceinline__ void tc_commit2_mc(uint32_t bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(bar), "h"(mask) : "memory");
}
__device__ __forceinline__ void tc_mma2_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum) : "memory");
}

// Pair-CTA variant of gemm_nn_tc_kernel (launched as clusters of 2 = one CTA pair on a TPC). The pair owns a 256-row M tile:
// the CTA of cluster rank r holds rows [128 r, 128 r + 128) of A (raw + lo tiles, split by its own splitter warps) and HALF
// of every weight tile (rows [r BN/2, (r+1) BN/2) of the K-major B_hi / B_lo tiles); one thread of the leader CTA (rank 0)
// issues tcgen05.mma.cta_group::2 (M = 256, N = BN), which reads A from each CTA's own shared memory and each half of B once
// for both tensor cores, so the weight tiles cost half the TMA writes and half the operand reads per SM. Accumulators: rows
// of the CTA's M half in its own TMEM. Barriers: every CTA has its own full / empty / tfull; conv and tempty live in the
// leader (one lane per peer warp arrives remotely, cluster-scope release / acquire); the leader's commits are multicast to both CTAs.
__global__ void __launch_bounds__(TC_THREADS, 1)
gemm_nn_tc2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmBhi,
                   const __grid_constant__ CUtensorMap tmBlo, const __grid_constant__ CUtensorMap tmC, const TcParams p) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bars[3 * TC_MAX_STAGES + 4];
    __shared__ uint32_t tmem_slot;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t crank = cluster_ctarank();
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const int b_rows = p.BN / 2;
    const uint32_t b_half = (uint32_t)b_rows * 128u;
    const uint32_t stage_bytes = 2u * TC_A_TILE + 2u * b_half;
    auto a_hi = [&](int s) { return base + (uint32_t)s * stage_bytes; };
    auto a_lo = [&](int s) { return base + (uint32_t)s * stage_bytes + TC_A_TILE; };
    auto b_hi = [&](int s) { return base + (uint32_t)s * stage_bytes + 2u * TC_A_TILE; };
    auto b_lo = [&](int s) { return base + (uint32_t)s * stage_bytes + 2u * TC_A_TILE + b_half; };
    const uint32_t bar0 = smem_u32(bars);
    auto full = [&](int s) { return bar0 + 8u * s; };
    auto conv = [&](int s) { return bar0 + 8u * (TC_MAX_STAGES + s); };
    auto empty = [&](int s) { return bar0 + 8u * (2 * TC_MAX_STAGES + s); };
    auto tfull = [&](int a) { return bar0 + 8u * (3 * TC_MAX_STAGES + a); };
    auto tempty = [&](int a) { return bar0 + 8u * (3 * TC_MAX_STAGES + 2 + a); };

    const int num_kb = (p.K + TC_BK - 1) / TC_BK;
    const long m_pairs = (p.M + 2 * TC_BM - 1) / (2 * TC_BM);
    const long total = m_pairs * p.n_tiles_n;
    const long first = blockIdx.x / 2, stride = gridDim.x / 2;

    if (threadIdx.x == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmBhi) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmBlo) : "memory");
        for (int s = 0; s < TC_MAX_STAGES; ++s) { mbar_init(full(s), 1); mbar_init(conv(s), 8); mbar_init(empty(s), 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(tfull(a), 1); mbar_init(tempty(a), 8); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = tmem_slot;

    if (warp == 0) {
        if (lane == 0) {                                           // ---- TMA producer (both CTAs, own halves)
            uint32_t it = 0;
            for (long tile = first; tile < total; tile += stride) {
                const int m0 = (int)((tile / p.n_tiles_n) * 2 + crank) * TC_BM;
                const int n0 = (int)(tile % p.n_tiles_n) * p.BN + (int)crank * b_rows;
                for (int kb = 0; kb < num_kb; ++kb, ++it) {
                    const int s = it % p.stages;
                    const uint32_t ph = (it / p.stages) & 1u;
                    mbar_wait_cluster(empty(s), ph ^ 1u);           // the leader's MMAs have released this stage in both CTAs
                    mbar_arrive_expect_tx(full(s), TC_A_TILE + 2u * b_half);
                    tma_load_2d(a_hi(s), &tmA, full(s), kb * TC_BK, m0);
                    tma_load_2d(b_hi(s), &tmBhi, full(s), kb * TC_BK, n0);
                    tma_load_2d(b_lo(s), &tmBlo, full(s), kb * TC_BK, n0);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0 && crank == 0) {                             // ---- MMA issuer (leader CTA only)
            const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(p.BN >> 3) << 17) | ((uint32_t)((2 * TC_BM) >> 4) << 24);
            uint32_t it = 0, tl = 0;
            for (long tile = first; tile < total; tile += stride, ++tl) {
                const uint32_t acc = tl & 1u, aph = (tl >> 1) & 1u;
                mbar_wait_cluster(tempty(acc), aph ^ 1u);           // both CTAs' epilogues have drained this accumulator
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * 256u;
                for (int kb = 0; kb < num_kb; ++kb, ++it) {
                    const int s = it % p.stages;
                    const uint32_t ph = (it / p.stages) & 1u;
                    mbar_wait(full(s), ph);                         // my tiles landed
                    mbar_wait_cluster(conv(s), ph);                 // both CTAs (4 + 4 splitter warps): tiles landed, A_lo written
                    tc_fence_after();
                    const uint64_t dah = make_kmajor_sw128_desc(a_hi(s)), dal = make_kmajor_sw128_desc(a_lo(s));
                    const uint64_t dbh = make_kmajor_sw128_desc(b_hi(s)), dbl = make_kmajor_sw128_desc(b_lo(s));
#pragma unroll
                    for (int ks = 0; ks < TC_BK / 8; ++ks) {
                        if (kb * TC_BK + ks * 8 >= p.K) break;
                        const uint64_t o = (uint64_t)(2 * ks);
                        tc_mma2_tf32(d_tmem, dal + o, dbh + o, idesc, (kb | ks) != 0);
                        tc_mma2_tf32(d_tmem, dah + o, dbl + o, idesc, 1u);
                        tc_mma2_tf32(d_tmem, dah + o, dbh + o, idesc, 1u);
                    }
                    tc_commit2_mc(empty(s), (uint16_t)3);           // frees the stage in both CTAs
                }
                tc_commit2_mc(tfull(acc), (uint16_t)3);             // accumulators complete -> both epilogues
            }
        }
    } else if (warp < 6) {                                         // ---- splitter (both CTAs): A_lo beside the raw tile
        const int t = threadIdx.x - 64;
        uint32_t it = 0;
        for (long tile = first; tile < total; tile += stride) {
            for (int kb = 0; kb < num_kb; ++kb, ++it) {
                const int s = it % p.stages;
                const uint32_t ph = (it / p.stages) & 1u;
                mbar_wait(full(s), ph);
                const uint32_t hi0 = a_hi(s), lo0 = a_lo(s);
#pragma unroll
                for (int i = 0; i < TC_A_TILE / 16 / 128; ++i) {
                    const uint32_t off = (uint32_t)(t + 128 * i) * 16u;
                    float4 x;
                    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(x.x), "=f"(x.y), "=f"(x.z), "=f"(x.w) : "r"(hi0 + off));
                    float4 l;
                    l.x = x.x - __uint_as_float(__float_as_uint(x.x) & 0xffffe000u);
                    l.y = x.y - __uint_as_float(__float_as_uint(x.y) & 0xffffe000u);
                    l.z = x.z - __uint_as_float(__float_as_uint(x.z) & 0xffffe000u);
                    l.w = x.w - __uint_as_float(__float_as_uint(x.w) & 0xffffe000u);
                    asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(lo0 + off), "f"(l.x), "f"(l.y), "f"(l.z), "f"(l.w) : "memory");
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncwarp();                                       // one cluster-scope release per warp, not per thread
                if (lane == 0) mbar_arrive_remote(conv(s), 0u);     // (the per-thread form stalled the splitters on membar)
            }
        }
    } else {                                                       // ---- epilogue (warps 6..9, both CTAs): TMEM -> smem -> TMA
        const int q = warp & 3;
        const uint32_t stg0 = base + (uint32_t)p.stages * stage_bytes + (uint32_t)q * 8192u;
        uint32_t tl = 0, sb = 0;
        for (long tile = first; tile < total; tile += stride, ++tl) {
            const uint32_t acc = tl & 1u, aph = (tl >> 1) & 1u;
            const int row0 = (int)((tile / p.n_tiles_n) * 2 + crank) * TC_BM + q * 32;
            const int n0 = (int)(tile % p.n_tiles_n) * p.BN;
            mbar_wait_cluster(tfull(acc), aph);
            tc_fence_after();
            // A warp whose 32 rows lie past the last row of C has nothing to store, and it must not touch its staging buffers:
            // it commits no bulk group, so `wait_group.read 1` would keep admitting the LAST store of the previous tile as
            // the one allowed reader while its buffer is rewritten with this tile's zeros (lost C += rows; found by
            // test_gemm_nn[20000-52-416]: M tiles 156 = 2 x 148 CTAs + partial last tile).
            for (int c0 = 0; c0 < p.BN && row0 < p.M; c0 += 32) {
                if (n0 + c0 >= p.N) break;
                uint32_t r[32];
                const uint32_t taddr = tmem_base + acc * 256u + (uint32_t)c0 + ((uint32_t)(q * 32) << 16);
                asm volatile(
                    "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
                    "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
                    : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                      "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
                      "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
                      "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                    : "r"(taddr));
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if (p.act == 2) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) r[j] = __float_as_uint(tanhf(__uint_as_float(r[j])));
                } else if (p.act) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) r[j] = __float_as_uint(tc_elu(__uint_as_float(r[j])));
                }
                if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
                __syncwarp();
                const uint32_t stg = stg0 + sb * 4096u;
                const uint32_t rowaddr = stg + (uint32_t)lane * 128u;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const uint32_t a = rowaddr + (uint32_t)((j ^ (lane & 7)) << 4);
                    asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(a), "r"(r[4 * j]), "r"(r[4 * j + 1]),
                                 "r"(r[4 * j + 2]), "r"(r[4 * j + 3]) : "memory");
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncwarp();
                if (lane == 0 && row0 < p.M) {
                    if (p.accumulate)
                        asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%1, %2}], [%3];"
                                     ::"l"(&tmC), "r"(n0 + c0), "r"(row0), "r"(stg) : "memory");
                    else
                        asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group [%0, {%1, %2}], [%3];"
                                     ::"l"(&tmC), "r"(n0 + c0), "r"(row0), "r"(stg) : "memory");
                    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                }
                sb ^= 1u;
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_remote(tempty(acc), 0u);
        }
        if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// Bt_hi/Bt_lo[n, k] = split(B[k, n]) : transposed (K-major), zero padded to ldt
__global__ void tc_prepare_b_kernel(const float* __restrict__ B, long ldb, int K, int N, float* __restrict__ hi,
                                    float* __restrict__ lo, int ldt) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long)N * ldt) return;
    const int n = (int)(i / ldt), k = (int)(i % ldt);
    const float x = k < K ? B[(long)k * ldb + n] : 0.f;
    const float h = __uint_as_float(__float_as_uint(x) & 0xffffe000u);
    hi[i] = h;
    lo[i] = x - h;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

// 2-D fp32 tensor [rows, cols] with row stride ld (floats); box = [box_rows, 32 cols], 128B swizzle, OOB -> 0
int make_map(CUtensorMap* tm, const float* ptr, long rows, long cols, long ld, int box_rows,
             CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) { set_error("gemm_tc: cuTensorMapEncodeTiled unavailable"); return 3; }
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
    cuuint32_t box[2] = {(cuuint32_t)TC_BK, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    const CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(ptr), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("gemm_tc: cuTensorMapEncodeTiled failed (%d)", (int)r); return 3; }
    return 0;
}
}  // namespace

int gemm_tc_ldt(int K) { return (K + 3) / 4 * 4; }

// SPK_TC_CLUSTER=2 enables 2-CTA clusters that share every weight tile by TMA multicast. EXPERIMENTAL, off by default:
// measured on B200 it gains only 2-3 % on the 416-wide products (the kernel is bound by shared-memory bandwidth, not by the
// L2 -> SM re-stream of the weights: profiles/README.md, round 2) and the C += (TMA reduce-add) epilogue lost updates on
// short-K shapes in this mode, so it is never combined with `accumulate`.
static int tc_cluster() {
    const char* e = getenv("SPK_TC_CLUSTER");
    return (e && e[0] == '2') ? 2 : 1;
}

// SPK_TC_PAIR=1 selects the pair-CTA (cta_group::2) kernel. EXPERIMENTAL, off by default: correct (tests/test_gpu_parity.py
// runs the GEMM tests in this mode too) and it cuts the L2 -> SM operand traffic by 39 % (ncu: 16.1 -> 9.9 GB on
// [2M,200]x[200,416]), but it is 5-40 % SLOWER on every product of the step: 3xTF32 re-reads each weight half 12 times per
// k-block and in pair mode half of those reads cross the SM-to-SM path (profiles/README.md, round 2). Read on every call so
// tests can toggle it.
static int tc_pair() {
    const char* e = getenv("SPK_TC_PAIR");
    return (e && e[0] == '1') ? 1 : 0;
}

// SPK_TC_RAW_HI=0 restores the explicit hi rewrite in the splitter (default: the raw tile is the hi operand)
static int tc_raw_hi() {
    static int v = -1;
    if (v < 0) { const char* e = getenv("SPK_TC_RAW_HI"); v = (e && e[0] == '0') ? 0 : 1; }
    return v;
}

int gemm_nn_tc_supported(const float* A, long lda, long M, int N, int K) {
    return M >= 1 && N >= 1 && K >= 1 && (lda % 4 == 0) && ((reinterpret_cast<uintptr_t>(A) & 15) == 0) && lda >= K;
}

// workspace: 2 * N * ldt floats for the split / transposed weights
int gemm_nn_tc(const float* A, long lda, const float* B, long ldb, float* C, long ldc, long M, int N, int K,
               int accumulate, float* workspace, cudaStream_t s, int act) {
    const int ldt = gemm_tc_ldt(K);
    float* bhi = workspace;
    float* blo = workspace + (long)N * ldt;
    const long nb = (long)N * ldt;
    tc_prepare_b_kernel<<<(unsigned)((nb + 255) / 256), 256, 0, s>>>(B, ldb, K, N, bhi, blo, ldt);
    if (int rc = check_launch("tc_prepare_b")) return rc;

    const int n_tiles_n = (N + 255) / 256;
    // one N tile: multiple of 16 columns (UMMA N); several: multiple of 32 so that the 32-column store boxes of the
    // epilogue never reach into the neighbouring tile
    const int bn_round = n_tiles_n > 1 ? 32 : 16;
    int BN = ((N + n_tiles_n - 1) / n_tiles_n + bn_round - 1) / bn_round * bn_round;
    if (BN < 16) BN = 16;
    const int b_tile = BN * 128;
    const int stage_bytes = 2 * TC_A_TILE + 2 * b_tile;
    const int c_vec = (ldc % 4 == 0) && ((reinterpret_cast<uintptr_t>(C) & 15) == 0);
    // the TMA epilogue writes a row's last box up to the next 16-byte boundary: with N % 4 != 0 it reaches the floats past
    // column N, outside the caller's view (seen on a B200: C += put NaN there in rows whose product is NaN)
    const int c_tma = c_vec && (N % 4 == 0) && !(act && accumulate);
    const int staging = c_tma ? 4 * 8192 : 0;                       // 4 epilogue warps x 2 x [32 x 32] fp32
    int stages = (225 * 1024 - 1024 - staging) / stage_bytes;
    if (stages > TC_MAX_STAGES) stages = TC_MAX_STAGES;
    if (stages < 1) { set_error("gemm_tc: tile does not fit shared memory"); return 3; }
    const int smem = stages * stage_bytes + staging + 1024;

    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long m_tiles = (M + TC_BM - 1) / TC_BM;
    // clusters of 2 share each weight tile (half the L2 -> SM traffic of the re-streamed weights); worth it once every SM
    // has work either way
    // pair-CTA kernel (M = 256 per CTA pair, each weight tile split over the pair): needs the TMA epilogue, the raw tile
    // as hi operand, BN/2 a multiple of 8 rows, and enough tiles that every SM has work either way
    const bool pair = tc_pair() && c_tma && tc_raw_hi() && (BN % 16 == 0) && m_tiles * n_tiles_n >= 2L * sms;
    if (pair) {
        const int half_tile = BN / 2 * 128;
        const int stage2 = 2 * TC_A_TILE + 2 * half_tile;
        int stages2 = (225 * 1024 - 1024 - staging) / stage2;
        if (stages2 > TC_MAX_STAGES) stages2 = TC_MAX_STAGES;
        const int smem2 = stages2 * stage2 + staging + 1024;
        CUtensorMap tA, tBh, tBl, tC;
        if (int rc = make_map(&tA, A, M, K, lda, TC_BM)) return rc;
        if (int rc = make_map(&tBh, bhi, N, K, ldt, BN / 2)) return rc;
        if (int rc = make_map(&tBl, blo, N, K, ldt, BN / 2)) return rc;
        if (int rc = make_map(&tC, C, M, N, ldc, 32)) return rc;
        TcParams q = {};
        q.C = C; q.ldc = ldc; q.M = M; q.N = N; q.K = K; q.BN = BN; q.n_tiles_n = n_tiles_n; q.stages = stages2;
        q.accumulate = accumulate; q.act = act; q.c_vec = c_vec; q.c_tma = 1; q.raw_hi = 1; q.cs = 2;
        static SmemLimit lim2;
        if (lim2.ensure(gemm_nn_tc2_kernel, 226 * 1024) != cudaSuccess) {
            set_error("gemm_tc: cannot raise dynamic shared memory limit");
            (void)cudaGetLastError();
            return 3;
        }
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)sms / 2 * 2); cfg.blockDim = dim3(TC_THREADS); cfg.dynamicSmemBytes = (size_t)smem2; cfg.stream = s;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        static int pairs_resident[64] = {};
        int nc = (dev >= 0 && dev < 64) ? pairs_resident[dev] : 0;
        if (nc == 0) {
            if (cudaOccupancyMaxActiveClusters(&nc, gemm_nn_tc2_kernel, &cfg) != cudaSuccess || nc < 1) { (void)cudaGetLastError(); nc = sms / 4; }
            if (dev >= 0 && dev < 64) pairs_resident[dev] = nc;
        }
        const long pair_tiles = ((m_tiles + 1) / 2) * n_tiles_n;
        const long np = pair_tiles < nc ? pair_tiles : nc;
        cfg.gridDim = dim3((unsigned)(2 * np));
        (void)cudaLaunchKernelEx(&cfg, gemm_nn_tc2_kernel, tA, tBh, tBl, tC, q);
        return check_launch("gemm_nn_tc2");
    }
    const int cs = (tc_cluster() == 2 && !accumulate && m_tiles * n_tiles_n >= 2L * sms) ? 2 : 1;

    CUtensorMap tmA, tmBhi, tmBlo, tmC;
    if (int rc = make_map(&tmA, A, M, K, lda, TC_BM)) return rc;
    if (int rc = make_map(&tmBhi, bhi, N, K, ldt, BN / cs)) return rc;
    if (int rc = make_map(&tmBlo, blo, N, K, ldt, BN / cs)) return rc;
    if (c_tma) { if (int rc = make_map(&tmC, C, M, N, ldc, 32)) return rc; }
    else tmC = tmA;

    TcParams p = {};
    p.C = C; p.ldc = ldc; p.M = M; p.N = N; p.K = K; p.BN = BN; p.n_tiles_n = n_tiles_n; p.stages = stages;
    p.accumulate = accumulate; p.act = act;
    p.c_vec = c_vec; p.c_tma = c_tma; p.raw_hi = tc_raw_hi(); p.cs = cs;
    static SmemLimit lim;
    if (lim.ensure(gemm_nn_tc_kernel<false>, 226 * 1024) != cudaSuccess) {
        set_error("gemm_tc: cannot raise dynamic shared memory limit");
        (void)cudaGetLastError();
        return 3;
    }
    const long total = ((m_tiles + cs - 1) / cs) * n_tiles_n * cs;      // CTAs' worth of tiles
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)sms / cs * cs); cfg.blockDim = dim3(TC_THREADS); cfg.dynamicSmemBytes = (size_t)smem; cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)cs; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    long resident = sms;                                                // persistent kernel: exactly one wave of CTAs
    if (cs > 1) {
        // a GPC with an odd number of free SMs cannot host a whole pair: ask how many clusters are co-resident (cached per
        // device: 1 CTA per SM at this shared-memory size, so the answer does not depend on the shape)
        static int clusters[64] = {};
        int nc = (dev >= 0 && dev < 64) ? clusters[dev] : 0;
        if (nc == 0) {
            if (cudaOccupancyMaxActiveClusters(&nc, gemm_nn_tc_kernel<false>, &cfg) != cudaSuccess || nc < 1) { (void)cudaGetLastError(); nc = sms / cs / 2; }
            if (dev >= 0 && dev < 64) clusters[dev] = nc;
        }
        resident = (long)nc * cs;
    }
    unsigned grid = (unsigned)(total < resident ? total : resident);
    grid = grid / cs * cs;
    if (grid < (unsigned)cs) grid = (unsigned)cs;
    cfg.gridDim = dim3(grid);
    (void)cudaLaunchKernelEx(&cfg, gemm_nn_tc_kernel<false>, tmA, tmBhi, tmBlo, tmC, p);
    return check_launch("gemm_nn_tc");
}


// ------------------------------------------------------------------------------------------------
// TN product on the tensor cores:  D[Ka, Nb] = sum_m X[m, Ka] * G[m, Nb]   (weight gradients, K5)
// Both operands are activations stored with the reduction index m as the ROW index, i.e. "MN-major"
// for the MMA: TMA lands [32 m-rows x 32 columns] boxes (128B swizzle with 32B atomicity, the only
// MN-major layout the tensor core takes for 32-bit operands); the UMMA descriptors use the MN-major
// canonical layout (LBO = distance between 32-column chunks, SBO = distance between 4-row groups)
// and the instruction descriptor sets a_major = b_major = MN. Both tiles are split hi/lo in
// shared memory by the splitter warps. One CTA = one (Ka-tile, Nb-tile, m-split); the per-split
// partials are added in split order by tn_reduce (deterministic).
// ------------------------------------------------------------------------------------------------
namespace {

constexpr int TN_BKM = 32;                     // m rows per pipeline stage (4 MMA K-steps)
constexpr int TN_CHUNK = TN_BKM * 128;         // one [32 rows x 32 cols] box = 4 KB
constexpr int TN_ACH = 4;                      // A chunks: 4 x 32 = 128 = UMMA M

__device__ __forceinline__ uint64_t make_mnmajor_sw128_desc(uint32_t saddr) {
    // 32-bit MN-major operands must use the 128B swizzle with 32B atomicity (cute::UMMA::LayoutType::SWIZZLE_128B_BASE32B,
    // Swizzle<2,5,2>): rows of 128 B, swizzle period 4 rows, canonical layout ((4,8,m),(4,k)) : ((1,4,LBO),(32,SBO)) floats.
    const uint32_t lo = ((saddr >> 4) & 0x3fffu) | ((uint32_t)(TN_CHUNK >> 4) << 16);   // start | LBO: next 32-col chunk
    const uint32_t hi = (512u >> 4) | (1u << 14) | (1u << 29);                         // SBO: next 4-row group | v1 | SW128_BASE32B
    return ((uint64_t)hi << 32) | lo;
}

struct TnParams {
    float* part; long M; int Ka; int Nb; int BN; int n_tiles_n; int n_tiles_k; int splits; long m_per_split; int stages;
    int raw_hi;
    const int* task_row0;                       // grouped kernel only: split z covers rows [task_row0[z], task_row1[z]) and
    const int* task_row1;                       // runs when z < *n_tasks
    const int* n_tasks;
};

// Decoupled rings: the raw tiles (TMA destination; read by the MMA as the "hi" operands) live in a ring of
// p.stages slots so the DRAM latency of both streamed operands is covered, the split-off "lo" tiles in a
// 2-slot ring written by the splitter warps right before the MMA consumes them.
constexpr int TN_LO_SLOTS = 2;
constexpr int TN_SPLIT_WARPS = 8;
constexpr int TN_THREADS = (2 + TN_SPLIT_WARPS + 4) * 32;      // TMA, MMA, splitters, epilogue

template <bool GROUPED>
__global__ void __launch_bounds__(TN_THREADS, 1)
gemm_tn_tc_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmG, const TnParams p) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bars[2 * TC_MAX_STAGES + 2 * TN_LO_SLOTS + 1];
    __shared__ uint32_t tmem_slot;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const int nbc = p.BN / 32;                                     // B chunks
    const uint32_t half = (uint32_t)(TN_ACH + nbc) * TN_CHUNK;     // one slot: A chunks, then B chunks
    const uint32_t b_off = TN_ACH * TN_CHUNK;
    auto raw = [&](int s) { return base + (uint32_t)s * half; };
    auto lo = [&](int l) { return base + (uint32_t)(p.stages + l) * half; };
    const uint32_t bar0 = smem_u32(bars);
    auto full = [&](int s) { return bar0 + 8u * s; };                                       // TMA -> splitter, MMA
    auto rawfree = [&](int s) { return bar0 + 8u * (TC_MAX_STAGES + s); };                  // MMA commit -> TMA
    auto conv = [&](int l) { return bar0 + 8u * (2 * TC_MAX_STAGES + l); };                 // splitter -> MMA
    auto lofree = [&](int l) { return bar0 + 8u * (2 * TC_MAX_STAGES + TN_LO_SLOTS + l); }; // MMA commit -> splitter
    const uint32_t tfull = bar0 + 8u * (2 * TC_MAX_STAGES + 2 * TN_LO_SLOTS);

    const int tile = blockIdx.x % (p.n_tiles_k * p.n_tiles_n);
    const int split = blockIdx.x / (p.n_tiles_k * p.n_tiles_n);
    if (GROUPED && split >= *p.n_tasks) return;                    // (the grid is sized for the largest task count)
    const int ka0 = (tile / p.n_tiles_n) * 128, nb0 = (tile % p.n_tiles_n) * p.BN;
    const long mbeg = GROUPED ? (long)p.task_row0[split] : (long)split * p.m_per_split;
    long mend = GROUPED ? (long)p.task_row1[split] : mbeg + p.m_per_split;
    if (mend > p.M) mend = p.M;
    const int num_kb = mend > mbeg ? (int)((mend - mbeg + TN_BKM - 1) / TN_BKM) : 0;

    if (threadIdx.x == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmX) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmG) : "memory");
        for (int s = 0; s < TC_MAX_STAGES; ++s) { mbar_init(full(s), 1); mbar_init(rawfree(s), 1); }
        for (int l = 0; l < TN_LO_SLOTS; ++l) { mbar_init(conv(l), TN_SPLIT_WARPS * 32); mbar_init(lofree(l), 1); }
        mbar_init(tfull, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"(256u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_slot;

    if (warp == 0) {
        if (lane == 0) {                                           // ---- TMA producer
            for (int kb = 0; kb < num_kb; ++kb) {
                const int s = kb % p.stages;
                const uint32_t ph = (kb / p.stages) & 1u;
                mbar_wait(rawfree(s), ph ^ 1u);
                mbar_arrive_expect_tx(full(s), half);
                // rows beyond `mend` belong to the next split: they are loaded and zeroed by the splitter
                const int m0 = (int)(mbeg + (long)kb * TN_BKM);
                for (int c = 0; c < TN_ACH; ++c) tma_load_2d(raw(s) + c * TN_CHUNK, &tmX, full(s), ka0 + 32 * c, m0);
                for (int c = 0; c < nbc; ++c) tma_load_2d(raw(s) + b_off + c * TN_CHUNK, &tmG, full(s), nb0 + 32 * c, m0);
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {                                           // ---- MMA issuer
            const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (1u << 15) | (1u << 16) |
                                   ((uint32_t)(p.BN >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
            for (int kb = 0; kb < num_kb; ++kb) {
                const int s = kb % p.stages, l = kb % TN_LO_SLOTS;
                mbar_wait(full(s), (kb / p.stages) & 1u);
                mbar_wait(conv(l), (kb / TN_LO_SLOTS) & 1u);
                tc_fence_after();
                const uint64_t dah = make_mnmajor_sw128_desc(raw(s)), dal = make_mnmajor_sw128_desc(lo(l));
                const uint64_t dbh = make_mnmajor_sw128_desc(raw(s) + b_off), dbl = make_mnmajor_sw128_desc(lo(l) + b_off);
#pragma unroll
                for (int ks = 0; ks < TN_BKM / 8; ++ks) {
                    const uint64_t o = (uint64_t)(ks * (1024 >> 4));     // next 8-row group
                    tc_mma_tf32(tmem_base, dal + o, dbh + o, idesc, (kb | ks) != 0);
                    tc_mma_tf32(tmem_base, dah + o, dbl + o, idesc, 1u);
                    tc_mma_tf32(tmem_base, dah + o, dbh + o, idesc, 1u);
                }
                tc_commit(rawfree(s));
                tc_commit(lofree(l));
            }
            tc_commit(tfull);
        }
    } else if (warp < 2 + TN_SPLIT_WARPS) {                        // ---- splitter: both tiles, raw -> (hi in place, lo)
        const int t = threadIdx.x - 64;
        const int n16 = (int)(half / 16);
        for (int kb = 0; kb < num_kb; ++kb) {
            const int s = kb % p.stages, l = kb % TN_LO_SLOTS;
            mbar_wait(full(s), (kb / p.stages) & 1u);
            mbar_wait(lofree(l), ((kb / TN_LO_SLOTS) & 1u) ^ 1u);
            const uint32_t hi0 = raw(s), lo0 = lo(l);
            const long m0 = mbeg + (long)kb * TN_BKM;
            const int valid_rows = (int)(mend - m0 < TN_BKM ? mend - m0 : TN_BKM);   // rows past the split end count as 0
            for (int i = t; i < n16; i += TN_SPLIT_WARPS * 32) {
                const uint32_t off = (uint32_t)i * 16u;
                const int r = (i >> 3) & (TN_BKM - 1);             // row inside the 4 KB chunk (128 B per row)
                float4 x;
                asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(x.x), "=f"(x.y), "=f"(x.z), "=f"(x.w) : "r"(hi0 + off));
                if (r >= valid_rows) x = make_float4(0.f, 0.f, 0.f, 0.f);
                float4 h, l4;
                h.x = __uint_as_float(__float_as_uint(x.x) & 0xffffe000u); l4.x = x.x - h.x;
                h.y = __uint_as_float(__float_as_uint(x.y) & 0xffffe000u); l4.y = x.y - h.y;
                h.z = __uint_as_float(__float_as_uint(x.z) & 0xffffe000u); l4.z = x.z - h.z;
                h.w = __uint_as_float(__float_as_uint(x.w) & 0xffffe000u); l4.w = x.w - h.w;
                // rows past the split end must read as zero, so they are rewritten even in raw-hi mode
                if (!p.raw_hi || r >= valid_rows)
                    asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(hi0 + off), "f"(h.x), "f"(h.y), "f"(h.z), "f"(h.w) : "memory");
                asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(lo0 + off), "f"(l4.x), "f"(l4.y), "f"(l4.z), "f"(l4.w) : "memory");
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            mbar_arrive(conv(l));
        }
    } else {                                                       // ---- epilogue: TMEM -> partial[split][ka][nb]
        const int q = warp & 3;
        const int ka = ka0 + q * 32 + lane;
        float* prow = p.part + ((long)split * p.Ka + ka) * p.Nb;
        if (num_kb > 0) {
            mbar_wait(tfull, 0);
            tc_fence_after();
        }
        for (int c0 = 0; c0 < p.BN; c0 += 16) {
            uint32_t r[16];
            if (num_kb > 0) {
                const uint32_t taddr = tmem_base + (uint32_t)c0 + ((uint32_t)(q * 32) << 16);
                asm volatile(
                    "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                    : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                      "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                    : "r"(taddr));
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            } else {
#pragma unroll
                for (int j = 0; j < 16; ++j) r[j] = 0u;
            }
            if (ka < p.Ka) {
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const int nb = nb0 + c0 + j;
                    if (nb < p.Nb) prow[nb] = __uint_as_float(r[j]);
                }
            }
        }
        tc_fence_before();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(256u) : "memory");
    }
}

// 2-D fp32 tensor [rows, cols], box = [32 rows x 32 cols], 128B swizzle
int make_map_tn(CUtensorMap* tm, const float* ptr, long rows, long cols, long ld) {
    return make_map(tm, ptr, rows, cols, ld, TN_BKM, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B);
}

__global__ void tn_reduce_tc_kernel(const float* __restrict__ part, int splits, long elems, int Nb,
                                    float* __restrict__ C, long ldc, int accumulate) {
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= elems) return;
    float s = 0.f;
    for (int z = 0; z < splits; ++z) s += part[(long)z * elems + idx];     // fixed order
    float* c = C + (idx / Nb) * ldc + (idx % Nb);
    *c = accumulate ? *c + s : s;
}

struct TnPlan { int n_tiles_k, n_tiles_n, BN, splits, stages, smem; long m_per_split; };

TnPlan tn_plan(long M, int Ka, int Nb) {
    TnPlan pl;
    pl.n_tiles_k = (Ka + 127) / 128;
    pl.n_tiles_n = (Nb + 255) / 256;
    pl.BN = ((Nb + pl.n_tiles_n - 1) / pl.n_tiles_n + 31) / 32 * 32;
    const int tiles = pl.n_tiles_k * pl.n_tiles_n;
    long splits = (148 + tiles - 1) / tiles;
    const long max_by_m = (M + 1023) / 1024;
    if (splits > max_by_m) splits = max_by_m;
    if (splits < 1) splits = 1;
    long mps = (M + splits - 1) / splits;
    mps = (mps + TN_BKM - 1) / TN_BKM * TN_BKM;
    if (mps < TN_BKM) mps = TN_BKM;
    pl.splits = (int)((M + mps - 1) / mps);
    if (pl.splits < 1) pl.splits = 1;
    pl.m_per_split = mps;
    const int half = (TN_ACH + pl.BN / 32) * TN_CHUNK;              // one slot (A chunks + B chunks)
    pl.stages = (225 * 1024 - 1024) / half - TN_LO_SLOTS;           // raw slots next to the 2 lo slots
    if (pl.stages > TC_MAX_STAGES) pl.stages = TC_MAX_STAGES;
    if (pl.stages < 1) pl.stages = 1;
    pl.smem = (pl.stages + TN_LO_SLOTS) * half + 1024;
    return pl;
}
}  // namespace

int gemm_tn_tc_supported(const float* A, long lda, const float* B, long ldb, long M, int Ka, int Nb) {
    return M >= 1 && Ka >= 1 && Nb >= 1 && (lda % 4 == 0) && (ldb % 4 == 0) && lda >= Ka && ldb >= Nb &&
           ((reinterpret_cast<uintptr_t>(A) & 15) == 0) && ((reinterpret_cast<uintptr_t>(B) & 15) == 0);
}

long gemm_tn_tc_workspace_floats(long M, int Ka, int Nb) {
    const TnPlan pl = tn_plan(M, Ka, Nb);
    return (long)pl.splits * Ka * Nb;
}

int gemm_tn_tc(const float* A, long lda, const float* B, long ldb, float* C, long ldc, long M, int Ka, int Nb,
               int accumulate, float* workspace, cudaStream_t s) {
    const TnPlan pl = tn_plan(M, Ka, Nb);
    CUtensorMap tmX, tmG;
    if (int rc = make_map_tn(&tmX, A, M, Ka, lda)) return rc;
    if (int rc = make_map_tn(&tmG, B, M, Nb, ldb)) return rc;
    TnParams p = {};
    p.part = workspace; p.M = M; p.Ka = Ka; p.Nb = Nb; p.BN = pl.BN; p.n_tiles_n = pl.n_tiles_n; p.n_tiles_k = pl.n_tiles_k;
    p.splits = pl.splits; p.m_per_split = pl.m_per_split; p.stages = pl.stages; p.raw_hi = tc_raw_hi();
    static SmemLimit lim;
    if (lim.ensure(gemm_tn_tc_kernel<false>, 226 * 1024) != cudaSuccess) {
        set_error("gemm_tn_tc: cannot raise dynamic shared memory limit");
        (void)cudaGetLastError();
        return 3;
    }
    const unsigned grid = (unsigned)(pl.n_tiles_k * pl.n_tiles_n * pl.splits);
    gemm_tn_tc_kernel<false><<<grid, TN_THREADS, pl.smem, s>>>(tmX, tmG, p);
    if (int rc = check_launch("gemm_tn_tc")) return rc;
    const long elems = (long)Ka * Nb;
    tn_reduce_tc_kernel<<<(unsigned)((elems + 255) / 256), 256, 0, s>>>(workspace, pl.splits, elems, Nb, C, ldc, accumulate);
    return check_launch("tn_reduce_tc");
}

// ------------------------------------------------------------------------------------------------
// Grouped products for the relation-space projection of the GAT_sep_space variant (spk_ent2rel_*):
// rows grouped by relation, every group padded with zero rows to whole 128-row M tiles, group g
// multiplying by its own weight W[group_rel[g]]. Group count, tile table and task table live on the
// device; the host sizes grids and buffers for the worst case and never reads them back.
// ------------------------------------------------------------------------------------------------
namespace {

// Bt_hi / Bt_lo of every present group, stacked: row g * N + n, column k < ldt holds split(W[r][k-th element of the
// n-th output column]) = W[r * rstride + n * sn + k * sk] (zero for k >= K). sn = 1, sk = N reads W[r] as B [K, N]
// (transposed into K-major); sn = ldw, sk = 1 reads it as B^T, i.e. multiplies by W[r]^T (no transpose).
__global__ void tc_prepare_b_grouped_kernel(const float* __restrict__ W, long rstride, long sn, long sk, int K, int N,
                                            const int* __restrict__ group_rel, const int* __restrict__ n_groups,
                                            float* __restrict__ hi, float* __restrict__ lo, int ldt) {
    const long per = (long)N * ldt;
    const long total = (long)*n_groups * per;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        const long g = i / per, rem = i % per;
        const int n = (int)(rem / ldt), k = (int)(rem % ldt);
        const float x = k < K ? W[(long)group_rel[g] * rstride + n * sn + k * sk] : 0.f;
        const float h = __uint_as_float(__float_as_uint(x) & 0xffffe000u);
        hi[i] = h;
        lo[i] = x - h;
    }
}

// dW[r] = sum of the partials of group rel2group[r]'s tasks, in task order (zeros for a relation without rows)
__global__ void tn_reduce_grouped_kernel(const float* __restrict__ part, const int* __restrict__ rel2group,
                                         const int* __restrict__ task_ptr, long elems, int n_rel, float* __restrict__ C) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= elems * n_rel) return;
    const int r = (int)(i / elems);
    const long idx = i % elems;
    const int g = rel2group[r];
    float s = 0.f;
    if (g >= 0)
        for (int z = task_ptr[g]; z < task_ptr[g + 1]; ++z) s += part[(long)z * elems + idx];
    C[i] = s;
}

}  // namespace

int gemm_nn_tc_grouped(const float* A, long lda, long max_rows, const float* W, long rstride, long sn, long sk,
                       int N, int K, const int* group_rel, const int* n_groups, int max_groups, const int* tile_group,
                       const int* n_mtiles, float* C, long ldc, int act, float* workspace, cudaStream_t s) {
    const int ldt = gemm_tc_ldt(K);
    float* bhi = workspace;
    float* blo = workspace + (long)max_groups * N * ldt;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long nb = (long)max_groups * N * ldt;
    long pblocks = (nb + 255) / 256;
    if (pblocks > 8L * sms) pblocks = 8L * sms;
    tc_prepare_b_grouped_kernel<<<(unsigned)(pblocks > 0 ? pblocks : 1), 256, 0, s>>>(W, rstride, sn, sk, K, N, group_rel,
                                                                                     n_groups, bhi, blo, ldt);
    if (int rc = check_launch("tc_prepare_b_grouped")) return rc;

    // tile shape, epilogue and pipeline depth exactly as gemm_nn_tc, so a group's rows come out as that kernel gives them
    const int n_tiles_n = (N + 255) / 256;
    const int bn_round = n_tiles_n > 1 ? 32 : 16;
    int BN = ((N + n_tiles_n - 1) / n_tiles_n + bn_round - 1) / bn_round * bn_round;
    if (BN < 16) BN = 16;
    const int stage_bytes = 2 * TC_A_TILE + 2 * BN * 128;
    const int c_vec = (ldc % 4 == 0) && ((reinterpret_cast<uintptr_t>(C) & 15) == 0);
    const int c_tma = c_vec && (N % 4 == 0);
    const int staging = c_tma ? 4 * 8192 : 0;
    int stages = (225 * 1024 - 1024 - staging) / stage_bytes;
    if (stages > TC_MAX_STAGES) stages = TC_MAX_STAGES;
    if (stages < 1) { set_error("gemm_tc_grouped: tile does not fit shared memory"); return 3; }
    const int smem = stages * stage_bytes + staging + 1024;

    CUtensorMap tmA, tmBhi, tmBlo, tmC;
    if (int rc = make_map(&tmA, A, max_rows, K, lda, TC_BM)) return rc;
    if (int rc = make_map(&tmBhi, bhi, (long)max_groups * N, K, ldt, BN)) return rc;
    if (int rc = make_map(&tmBlo, blo, (long)max_groups * N, K, ldt, BN)) return rc;
    if (c_tma) { if (int rc = make_map(&tmC, C, max_rows, N, ldc, 32)) return rc; }
    else tmC = tmA;

    TcParams p = {};
    p.C = C; p.ldc = ldc; p.M = max_rows; p.N = N; p.K = K; p.BN = BN; p.n_tiles_n = n_tiles_n; p.stages = stages;
    p.accumulate = 0; p.act = act; p.c_vec = c_vec; p.c_tma = c_tma; p.raw_hi = tc_raw_hi(); p.cs = 1;
    p.tile_group = tile_group; p.n_mtiles = n_mtiles;
    static SmemLimit lim;
    if (lim.ensure(gemm_nn_tc_kernel<true>, 226 * 1024) != cudaSuccess) {
        set_error("gemm_tc_grouped: cannot raise dynamic shared memory limit");
        (void)cudaGetLastError();
        return 3;
    }
    const long max_tiles = (max_rows + TC_BM - 1) / TC_BM * n_tiles_n;
    const unsigned grid = (unsigned)(max_tiles < sms ? (max_tiles > 0 ? max_tiles : 1) : sms);
    gemm_nn_tc_kernel<true><<<grid, TC_THREADS, smem, s>>>(tmA, tmBhi, tmBlo, tmC, p);
    return check_launch("gemm_nn_tc_grouped");
}

long gemm_tn_tc_grouped_workspace_floats(int max_tasks, int Ka, int Nb) { return (long)max_tasks * Ka * Nb; }

int gemm_tn_tc_grouped(const float* A, long lda, const float* B, long ldb, long max_rows, int Ka, int Nb,
                       const int* task_row0, const int* task_row1, const int* n_tasks, int max_tasks,
                       const int* rel2group, const int* task_ptr, int n_rel, float* C, float* workspace, cudaStream_t s) {
    const TnPlan pl = tn_plan(max_rows, Ka, Nb);
    CUtensorMap tmX, tmG;
    if (int rc = make_map_tn(&tmX, A, max_rows, Ka, lda)) return rc;
    if (int rc = make_map_tn(&tmG, B, max_rows, Nb, ldb)) return rc;
    TnParams p = {};
    p.part = workspace; p.M = max_rows; p.Ka = Ka; p.Nb = Nb; p.BN = pl.BN; p.n_tiles_n = pl.n_tiles_n;
    p.n_tiles_k = pl.n_tiles_k; p.splits = max_tasks; p.m_per_split = 0; p.stages = pl.stages; p.raw_hi = tc_raw_hi();
    p.task_row0 = task_row0; p.task_row1 = task_row1; p.n_tasks = n_tasks;
    static SmemLimit lim;
    if (lim.ensure(gemm_tn_tc_kernel<true>, 226 * 1024) != cudaSuccess) {
        set_error("gemm_tn_tc_grouped: cannot raise dynamic shared memory limit");
        (void)cudaGetLastError();
        return 3;
    }
    if (max_tasks > 0) {
        const unsigned grid = (unsigned)(pl.n_tiles_k * pl.n_tiles_n * max_tasks);
        gemm_tn_tc_kernel<true><<<grid, TN_THREADS, pl.smem, s>>>(tmX, tmG, p);
        if (int rc = check_launch("gemm_tn_tc_grouped")) return rc;
    }
    const long elems = (long)Ka * Nb;
    tn_reduce_grouped_kernel<<<(unsigned)((elems * n_rel + 255) / 256), 256, 0, s>>>(workspace, rel2group, task_ptr, elems,
                                                                                     n_rel, C);
    return check_launch("tn_reduce_grouped");
}

}  // namespace spk
