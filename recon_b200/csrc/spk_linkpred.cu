// ConvKB link-prediction evaluation: filtered entity ranks (Corpus.get_validation_pred, GAT/create_batch.py:905-1199).
//   For every test row (h, r, t) the reference scores (c, r, t) and (h, r, c) for all entities c with batch_test, drops the
//   candidates that are known triples, puts the test triple first and reads its position after a descending sort. The
//   rank needs only a count, so the T x N score matrix never exists here:
//     count[i] = #{c in [0, N), c != true_i : s_c > s_true_i}         (spk_linkpred_count, a SIMT-GEMM-shaped pass)
//     count[i] -= #{distinct known c != true_i : s_c > s_true_i}      (spk_linkpred_filter, over the sorted key ranges)
//   with a > b meaning a > b or (isnan(a) && !isnan(b)) (torch.sort orders NaN as largest) and rank = 1 + count.
// Scores use the re-association of relation_scores: fc1([e_h | rel_r | e_t]) = A[h] + Bt[r] + C[t] + b1, AC = [A | C] one
// [N, 2D] table, so a pair vector v_i = C[t_i] + Bt[r_i] + b1 (head side) or A[h_i] + Bt[r_i] + b1 (tail side) meets every
// candidate row X[c] = A[c] or C[c]:  s_c = sum_d w2[d] * lrelu(X[c, d] + v_i[d])  (fc2's bias shifts a whole row: dropped).
// Bit identity: a filtered candidate's score must be the same float in the count pass and the filter pass, and s_true
// must come from the same arithmetic, or a subtraction could disagree with the count it corrects. Every score is therefore
// one sequential fp32 chain over d = 0..D-1 of lp_step (explicit _rn intrinsics: no contraction differences), used by all
// three kernels; lrelu(x) = max(x, slope * x), exact for 0 <= slope <= 1 (NaN stays NaN).
#include "../../include/spkbgat.h"
#include "spk_common.cuh"

namespace spk {
namespace {

constexpr int LP_MAX_D = 512;
constexpr int LP_BC = 128, LP_BK = 8;                    // candidates per CTA tile, k-chunk per pipeline stage
// Pair-tile heights of lp_count_kernel: a call with at most LP_NARROW_MAX pairs uses LP_BP_NARROW-row tiles, so a small
// test set (one relation group of the GAT_sep_space evaluation, usually 1-3 rows) does not pay for 128 padded pairs
// against all N candidates; larger calls use 128-row tiles, which reuse every staged candidate value 8x more often.
// Crossover measured with profiles/bench_linkpred_sep.py on a B200 (DESIGN.md section 9, N4b): n pairs as 16-row tiles
// cost 1.41 ms per 16 rows at N = 2M, D = 200, one 128-row tile 8.04 ms: 7.04 ms at 80 pairs, 8.44 ms at 96.
constexpr int LP_BP_WIDE = 128, LP_BP_NARROW = 16;
constexpr long LP_NARROW_MAX = 80;

__device__ __forceinline__ float lp_step(float acc, float x_c, float v, float w, float slope) {
    const float x = __fadd_rn(x_c, v);
    return __fmaf_rn(w, fmaxf(x, __fmul_rn(slope, x)), acc);
}
__device__ __forceinline__ bool lp_gt(float a, float b) { return a > b || (isnan(a) && !isnan(b)); }

// The per-candidate path: s = chain over d of lp_step(X row, v row). Plain loads: the prologue reads back the V row its
// own warp just wrote.
__device__ __forceinline__ float lp_score(const float* x, const float* v, const float* __restrict__ w2, int D, float slope) {
    float s = 0.f;
    for (int d = 0; d < D; ++d) s = lp_step(s, x[d], v[d], __ldg(w2 + d), slope);
    return s;
}

// One warp per test row: checks the ids, writes v_i, true_id (-1: skipped or invalid) and s_true, zeroes the count.
__global__ void __launch_bounds__(256)
lp_pairs_kernel(const float* __restrict__ AC, long ldac, long N, const float* __restrict__ Bt, long ldb, long R,
                const float* __restrict__ b1, const float* __restrict__ w2, float slope, int D,
                const long long* __restrict__ tri, const unsigned char* __restrict__ keep, long T, int side,
                float* __restrict__ V, long ldv, float* __restrict__ s_true, int* __restrict__ true_id,
                int* __restrict__ count, int* __restrict__ err) {
    const int lane = threadIdx.x & 31;
    const long i = (long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (i >= T) return;
    long long h = tri[3 * i], r = tri[3 * i + 1], t = tri[3 * i + 2];
    const bool bad = h < 0 || h >= N || t < 0 || t >= N || r < 0 || r >= R;
    if (bad) { if (lane == 0) atomicOr(err, 1); h = r = t = 0; }
    const long pid = side ? h : t, tid = side ? t : h;
    const float* P = AC + (side ? 0 : D) + pid * ldac;            // head side: C[t]; tail side: A[h]
    const float* B = Bt + r * ldb;
    float* v = V + i * ldv;
    for (int d = lane; d < D; d += 32) v[d] = __fadd_rn(__fadd_rn(__ldg(P + d), __ldg(B + d)), __ldg(b1 + d));
    __syncwarp();
    if (lane == 0) {
        const bool kept = !bad && (keep == nullptr || keep[i]);
        s_true[i] = kept ? lp_score(AC + (side ? D : 0) + tid * ldac, v, w2, D, slope) : 0.f;
        true_id[i] = kept ? (int)tid : -1;
        count[i] = 0;
    }
}

// Pair row of micro-tile row i of thread row ty in a BP-row tile: 128 rows: ty*4 + {0..3}, 64 + ty*4 + {0..3};
// narrower tiles: ty*(BP/16) + i.
template <int BP>
__device__ __forceinline__ int lp_pair_row(int i, int ty) {
    if constexpr (BP == 128) return i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4);
    else return ty * (BP / 16) + i;
}

// count[i] += #{c : c != true_i, s_c > s_true_i} for the candidate tiles blockIdx.y, blockIdx.y + gridDim.y, ...
// CTA tile: BP pairs x 128 candidates, 16 x 16 threads with a BP/16 x 8 register micro-tile each (rows lp_pair_row,
// columns tx*4 + {0..3}, 64 + tx*4 + {0..3}). V and X chunks of 8 k are staged through registers into double-buffered,
// transposed shared memory (the spk_gemm_simt.cu pipeline, carried across candidate tiles). After the last k chunk of a
// tile each thread compares its finished scores and counts in registers; the 16 threads of a pair row are summed by
// shuffles and added with one integer atomic per pair and CTA (order-independent, so counts are reproducible). Every
// score is the same lp_step chain whatever BP is, so every tile height gives the same counts.
template <int BP>
__global__ void __launch_bounds__(256, 2)
lp_count_kernel(const float* __restrict__ X, long ldx, long N, const float* __restrict__ V, long ldv,
                const float* __restrict__ w2, float slope, int D, const float* __restrict__ s_true,
                const int* __restrict__ true_id, long T, int x_vec, int v_vec, int* __restrict__ count) {
    static_assert(BP == 128 || (BP % 16 == 0 && BP / 16 <= 4), "pair tile: 128 rows, or 16 * (1..4)");
    constexpr int MI = BP / 16;                                   // micro-tile rows per thread
    __shared__ __align__(16) float Vs[2][LP_BK][BP + 4];
    __shared__ __align__(16) float Xs[2][LP_BK][LP_BC + 4];
    __shared__ float w2s[LP_MAX_D + LP_BK];
    const int tid = threadIdx.x;
    const int tx = tid & 15, ty = tid >> 4;
    const long p0 = (long)blockIdx.x * BP;

    int live = 0;
    for (int k = tid; k < BP; k += 256) live |= (p0 + k < T && true_id[p0 + k] >= 0);
    if (!__syncthreads_or(live)) return;                          // every row of this tile is skipped
    for (int d = tid; d < LP_MAX_D + LP_BK; d += 256) w2s[d] = d < D ? __ldg(w2 + d) : 0.f;

    float st[MI];
    int tr[MI], cnt[MI];
#pragma unroll
    for (int i = 0; i < MI; ++i) {
        const long p = p0 + lp_pair_row<BP>(i, ty);
        tr[i] = p < T ? true_id[p] : -1;
        st[i] = p < T ? s_true[p] : 0.f;
        cnt[i] = 0;
    }

    const long n_ct = (N + LP_BC - 1) / LP_BC;
    const long my_tiles = (n_ct - blockIdx.y + gridDim.y - 1) / gridDim.y;
    const int nk = (D + LP_BK - 1) / LP_BK;
    const long total = my_tiles * nk;
    const int l_row = tid >> 1, l_k = (tid & 1) * 4;              // loader: 128 rows x 8 k, 4 floats per thread
    const long c_step = (long)gridDim.y * LP_BC;
    long ld_c = (long)blockIdx.y * LP_BC;                         // next chunk to load: candidate tile row 0, k offset
    int ld_k = 0;
    float rx[4], rv[4];

    auto load = [&]() {
        const long c = ld_c + l_row, p = p0 + l_row;
        const int k = ld_k + l_k;
        if (c < N && x_vec && k + 3 < D) {
            const float4 q = ldg4(X + c * ldx + k);
            rx[0] = q.x; rx[1] = q.y; rx[2] = q.z; rx[3] = q.w;
        } else {
#pragma unroll
            for (int e = 0; e < 4; ++e) rx[e] = (c < N && k + e < D) ? __ldg(X + c * ldx + k + e) : 0.f;
        }
        if (BP == 128 || l_row < BP) {                             // the V tile has BP rows
            if (p < T && v_vec && k + 3 < D) {
                const float4 q = ldg4(V + p * ldv + k);
                rv[0] = q.x; rv[1] = q.y; rv[2] = q.z; rv[3] = q.w;
            } else {
#pragma unroll
                for (int e = 0; e < 4; ++e) rv[e] = (p < T && k + e < D) ? __ldg(V + p * ldv + k + e) : 0.f;
            }
        }
        ld_k += LP_BK;
        if (ld_k >= D) { ld_k = 0; ld_c += c_step; }
    };
    auto store = [&](int buf) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            Xs[buf][l_k + e][l_row] = rx[e];
            if (BP == 128 || l_row < BP) Vs[buf][l_k + e][l_row] = rv[e];
        }
    };

    float acc[MI][8];
#pragma unroll
    for (int i = 0; i < MI; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

    if (total > 0) { load(); store(0); }
    __syncthreads();
    long c0 = (long)blockIdx.y * LP_BC;                           // tile being computed
    int k0 = 0;
    for (long it = 0; it < total; ++it) {
        const int buf = (int)(it & 1);
        if (it + 1 < total) load();
        const int kn = min(LP_BK, D - k0);                        // the chain stops at d = D - 1 exactly
#pragma unroll
        for (int k = 0; k < LP_BK; ++k) {
            if (k < kn) {
                const float w = w2s[k0 + k];
                float vv[MI];
                if constexpr (BP == 128) {
                    const float4 v0 = *reinterpret_cast<const float4*>(&Vs[buf][k][ty * 4]);
                    const float4 v1 = *reinterpret_cast<const float4*>(&Vs[buf][k][64 + ty * 4]);
                    vv[0] = v0.x; vv[1] = v0.y; vv[2] = v0.z; vv[3] = v0.w;
                    vv[4] = v1.x; vv[5] = v1.y; vv[6] = v1.z; vv[7] = v1.w;
                } else {
#pragma unroll
                    for (int i = 0; i < MI; ++i) vv[i] = Vs[buf][k][ty * MI + i];
                }
                const float4 x0 = *reinterpret_cast<const float4*>(&Xs[buf][k][tx * 4]);
                const float4 x1 = *reinterpret_cast<const float4*>(&Xs[buf][k][64 + tx * 4]);
                const float xv[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
#pragma unroll
                for (int i = 0; i < MI; ++i)
#pragma unroll
                    for (int j = 0; j < 8; ++j) acc[i][j] = lp_step(acc[i][j], xv[j], vv[i], w, slope);
            }
        }
        k0 += LP_BK;
        if (k0 >= D) {                                            // candidate tile finished: compare, count, reset
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const long c = c0 + (j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4));
                const bool cv = c < N;
#pragma unroll
                for (int i = 0; i < MI; ++i) {
                    cnt[i] += (cv && c != tr[i] && lp_gt(acc[i][j], st[i])) ? 1 : 0;
                    acc[i][j] = 0.f;
                }
            }
            k0 = 0;
            c0 += c_step;
        }
        if (it + 1 < total) {
            store(buf ^ 1);
            __syncthreads();
        }
    }
#pragma unroll
    for (int i = 0; i < MI; ++i) {
        int c = cnt[i];
#pragma unroll
        for (int o = 1; o < 16; o <<= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
        const long p = p0 + lp_pair_row<BP>(i, ty);
        if (tx == 0 && tr[i] >= 0 && c) atomicAdd(count + p, c);   // tr[i] >= 0 implies p < T
    }
}

__device__ __forceinline__ long long lp_lower_bound(const long long* __restrict__ keys, long long m, long long key) {
    long long lo = 0, hi = m;
    while (lo < hi) {
        const long long mid = (lo + hi) >> 1;
        if (__ldg(keys + mid) < key) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// Key of the first candidate of row i: (base * R + r) * N with base = h (tail side) or t (head side, swapped keys).
__device__ __forceinline__ long long lp_range_base(const long long* __restrict__ tri, long i, int side, long long N, long long R) {
    const long long base = side ? tri[3 * i] : tri[3 * i + 2];
    return (base * R + tri[3 * i + 1]) * N;
}

// lo[i] = first key of row i's range, len[i] = its length (0 for a skipped row).
__global__ void __launch_bounds__(256)
lp_ranges_kernel(const long long* __restrict__ tri, long T, int side, long long N, long long R,
                 const int* __restrict__ true_id, const long long* __restrict__ keys, long long m,
                 long long* __restrict__ lo, long long* __restrict__ len) {
    const long i = (long)blockIdx.x * 256 + threadIdx.x;
    if (i >= T) return;
    long long a = 0, b = 0;
    if (true_id[i] >= 0) {
        const long long k0 = lp_range_base(tri, i, side, N, R);
        a = lp_lower_bound(keys, m, k0);
        b = lp_lower_bound(keys, m, k0 + N);
    }
    lo[i] = a;
    len[i] = b - a;
}

// off[0..T] = exclusive prefix sum of len (one CTA of 1024 threads, chunked; off[T] = total).
__global__ void __launch_bounds__(1024)
lp_scan_kernel(const long long* __restrict__ len, long T, long long* __restrict__ off) {
    __shared__ long long wsum[32];
    __shared__ long long carry_s;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    if (tid == 0) carry_s = 0;
    __syncthreads();
    for (long b = 0; b < T; b += 1024) {
        const long i = b + tid;
        const long long x = i < T ? len[i] : 0;
        long long s = x;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long y = __shfl_up_sync(0xffffffffu, s, o);
            if (lane >= o) s += y;
        }
        if (lane == 31) wsum[w] = s;
        __syncthreads();
        if (w == 0) {
            long long q = wsum[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const long long y = __shfl_up_sync(0xffffffffu, q, o);
                if (lane >= o) q += y;
            }
            wsum[lane] = q;                                       // inclusive warp totals
        }
        __syncthreads();
        const long long carry = carry_s;
        const long long incl = carry + (w ? wsum[w - 1] : 0) + s;
        if (i < T) off[i] = incl - x;
        __syncthreads();
        if (tid == 1023) carry_s = incl;
        __syncthreads();
    }
    if (tid == 0) off[T] = carry_s;
}

// One thread per (row, known candidate) item, flattened over the ranges so a hub range spreads over the whole grid.
// A distinct candidate c != true_i whose score beats s_true_i was counted by lp_count_kernel: take it back.
__global__ void __launch_bounds__(256)
lp_discount_kernel(const float* __restrict__ X, long ldx, long long N, long long R, const float* __restrict__ V, long ldv,
                   const float* __restrict__ w2, float slope, int D, const long long* __restrict__ tri, long T, int side,
                   const float* __restrict__ s_true, const int* __restrict__ true_id, const long long* __restrict__ keys,
                   const long long* __restrict__ lo, const long long* __restrict__ off, int* __restrict__ count,
                   int* __restrict__ err) {
    const long long total = off[T];
    for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < total; j += (long long)gridDim.x * blockDim.x) {
        long a = 0, b = T;                                        // row i: off[i] <= j < off[i + 1]
        while (b - a > 1) {
            const long mid = (a + b) >> 1;
            if (__ldg(off + mid) <= j) a = mid; else b = mid;
        }
        const long i = a;
        const long long k = __ldg(lo + i) + (j - __ldg(off + i));
        const long long key = __ldg(keys + k);
        if (k > 0 && __ldg(keys + k - 1) == key) continue;       // duplicate known triple: counted once
        const long long c = key - lp_range_base(tri, i, side, N, R);
        if (c < 0 || c >= N) { atomicOr(err, 2); continue; }
        if (c == true_id[i]) continue;
        const float s = lp_score(X + c * ldx, V + i * ldv, w2, D, slope);
        if (lp_gt(s, s_true[i])) atomicSub(count + i, 1);
    }
}

template <int BP>
int lp_launch_count(const float* X, long ldac, long n_ent, const float* V, long ldv, const float* w2, float slope, int D,
                    const float* s_true, const int* true_id, long n_pairs, int x_vec, int v_vec, int* count, cudaStream_t s) {
    int dev = 0, sms = 148, occ = 1;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, lp_count_kernel<BP>, 256, 0);
    const long gx = (n_pairs + BP - 1) / BP;
    const long n_ct = (n_ent + LP_BC - 1) / LP_BC;
    // one resident wave when the pair tiles allow it; the CTAs of one blockIdx.y walk the same candidate tiles together,
    // so each candidate row comes from HBM about once and from L2 for the other pair tiles
    long gy = (long)sms * (occ > 0 ? occ : 1) / gx;
    gy = gy < 1 ? 1 : (gy > n_ct ? n_ct : gy);
    if (gy > 65535) gy = 65535;
    if (gx > 0x7fffffffL) { set_error("linkpred_count: too many test rows"); return 1; }
    lp_count_kernel<BP><<<dim3((unsigned)gx, (unsigned)gy), 256, 0, s>>>(X, ldac, n_ent, V, ldv, w2, slope, D, s_true,
                                                                        true_id, n_pairs, x_vec, v_vec, count);
    return check_launch("linkpred_count");
}

int lp_check(const char* who, long long ldac, long long n_ent, long long n_rel, float slope, int D, int side) {
    if (D < 1 || ldac < 2LL * D || n_ent < 1 || n_ent >= (1LL << 31) - 1 || n_rel < 1 || (side != 0 && side != 1)) {
        set_error("%s: bad arguments", who);
        return 1;
    }
    if (D > LP_MAX_D) { set_error("%s: width %d exceeds %d", who, D, LP_MAX_D); return 2; }
    if (!(slope >= 0.f && slope <= 1.f)) { set_error("%s: LeakyReLU slope %g outside [0, 1]", who, (double)slope); return 1; }
    return 0;
}

}  // namespace
}  // namespace spk

using namespace spk;

extern "C" {

int spk_linkpred_count(const float* AC, int64_t ldac, int64_t n_ent, const float* Bt, int64_t ldb, int64_t n_rel,
                       const float* b1, const float* w2, float slope, int32_t D, const int64_t* triples,
                       const uint8_t* keep, int64_t n_pairs, int32_t side, float* V, int64_t ldv, float* s_true,
                       int32_t* true_id, int32_t* count, int32_t* err_flag, spk_stream_t stream) {
    if (int rc = lp_check("linkpred_count", ldac, n_ent, n_rel, slope, D, side)) return rc;
    if (ldb < D || ldv < D || !err_flag) { set_error("linkpred_count: bad arguments"); return 1; }
    if (n_pairs <= 0) return 0;
    const cudaStream_t s = (cudaStream_t)stream;
    const long long* tri = reinterpret_cast<const long long*>(triples);
    lp_pairs_kernel<<<(unsigned)((n_pairs + 7) / 8), 256, 0, s>>>(AC, (long)ldac, (long)n_ent, Bt, (long)ldb, (long)n_rel, b1,
                                                               w2, slope, D, tri, keep, (long)n_pairs, side, V, (long)ldv,
                                                               s_true, true_id, count, err_flag);
    if (int rc = check_launch("linkpred_pairs")) return rc;

    const float* X = AC + (side ? D : 0);
    const int x_vec = (ldac % 4 == 0) && ((reinterpret_cast<uintptr_t>(X) & 15) == 0);
    const int v_vec = (ldv % 4 == 0) && ((reinterpret_cast<uintptr_t>(V) & 15) == 0);
    if (n_pairs <= LP_NARROW_MAX)
        return lp_launch_count<LP_BP_NARROW>(X, ldac, n_ent, V, ldv, w2, slope, D, s_true, true_id, n_pairs, x_vec, v_vec,
                                             count, s);
    return lp_launch_count<LP_BP_WIDE>(X, ldac, n_ent, V, ldv, w2, slope, D, s_true, true_id, n_pairs, x_vec, v_vec, count, s);
}

int spk_linkpred_filter(const float* AC, int64_t ldac, int64_t n_ent, int64_t n_rel, const float* w2, float slope,
                        int32_t D, const int64_t* triples, int64_t n_pairs, int32_t side, const float* V, int64_t ldv,
                        const float* s_true, const int32_t* true_id, const int64_t* keys, int64_t n_keys, int64_t* work,
                        int32_t* count, int32_t* err_flag, spk_stream_t stream) {
    if (int rc = lp_check("linkpred_filter", ldac, n_ent, n_rel, slope, D, side)) return rc;
    if (ldv < D || !err_flag || (n_keys > 0 && (!keys || !work))) { set_error("linkpred_filter: bad arguments"); return 1; }
    if (n_pairs <= 0 || n_keys <= 0) return 0;
    const cudaStream_t s = (cudaStream_t)stream;
    const long long* tri = reinterpret_cast<const long long*>(triples);
    const long long* k = reinterpret_cast<const long long*>(keys);
    long long* lo = reinterpret_cast<long long*>(work);          // work = [lo: T | len: T | off: T + 1]
    long long* len = lo + n_pairs;
    long long* off = len + n_pairs;
    lp_ranges_kernel<<<(unsigned)((n_pairs + 255) / 256), 256, 0, s>>>(tri, (long)n_pairs, side, n_ent, n_rel, true_id, k,
                                                                       n_keys, lo, len);
    if (int rc = check_launch("linkpred_ranges")) return rc;
    lp_scan_kernel<<<1, 1024, 0, s>>>(len, (long)n_pairs, off);
    if (int rc = check_launch("linkpred_scan")) return rc;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    lp_discount_kernel<<<(unsigned)(sms * 8), 256, 0, s>>>(AC + (side ? D : 0), (long)ldac, n_ent, n_rel, V, (long)ldv, w2,
                                                           slope, D, tri, (long)n_pairs, side, s_true, true_id, k, lo, off,
                                                           count, err_flag);
    return check_launch("linkpred_discount");
}

}  // extern "C"
