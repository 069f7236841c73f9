// Relation-grouped row layout of the GAT_sep_space projection tanh(e . W_ent2rel[r]) (GAT_sep_space/models.py:316-320,
// GAT_sep_space/main.py:360-377), built on the device without a host round trip:
//
//   spk_ent2rel_keys       key[j] = relation of row j (n_rel for an id outside [0, n_rel): that row joins no group), val = j
//   (spk_sort_pairs + spk_segment_ptr: rows stably sorted by relation, segptr[r] = first row of relation r)
//   spk_ent2rel_plan       one CTA: groups = relations present, in id order; group g owns M tiles
//                          [group_tile0[g], group_tile0[g + 1]) of 128 rows (its rows, then zero rows up to the tile end)
//                          and the weight-gradient tasks [task_ptr[g], task_ptr[g + 1]) of up to tiles_per_task tiles;
//                          counts = {groups, M tiles, tasks}
//   spk_ent2rel_positions  pos[j] = padded row of input row j
//   spk_ent2rel_gather     out[p] = table[ids[src(p)]] for the real padded rows p, zero for the pad rows
//
// The grouped tcgen05 products that consume the layout are in spk_gemm_tc.cu (gemm_nn_tc_grouped, gemm_tn_tc_grouped).
#include "../../include/spkbgat.h"
#include "spk_common.cuh"
#include "spk_gemm.cuh"

namespace spk {

int gemm_nn_tc_grouped(const float* A, long lda, long max_rows, const float* W, long rstride, long sn, long sk,
                       int N, int K, const int* group_rel, const int* n_groups, int max_groups, const int* tile_group,
                       const int* n_mtiles, float* C, long ldc, int act, float* workspace, cudaStream_t s);
long gemm_tn_tc_grouped_workspace_floats(int max_tasks, int Ka, int Nb);
int gemm_tn_tc_grouped(const float* A, long lda, const float* B, long ldb, long max_rows, int Ka, int Nb,
                       const int* task_row0, const int* task_row1, const int* n_tasks, int max_tasks,
                       const int* rel2group, const int* task_ptr, int n_rel, float* C, float* workspace, cudaStream_t s);

namespace {

constexpr int E2R_TILE = 128;                 // = the M tile of the tcgen05 GEMMs
constexpr int PLAN_THREADS = 1024;

__global__ void ent2rel_keys_kernel(const long long* __restrict__ rel, long stride, long n_src, long n, int n_rel,
                                    int* __restrict__ keys, int* __restrict__ vals, int* __restrict__ err) {
    const long j = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const long long r = rel[(j % n_src) * stride];
    const bool ok = r >= 0 && r < n_rel;
    if (!ok) atomicOr(err, 1);
    keys[j] = ok ? (int)r : n_rel;
    vals[j] = (int)j;
}

// exclusive block scan of three counters; returns the block totals through tot[]
__device__ __forceinline__ void scan3(int v[3], int tot[3], int* sh) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int inc[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        int x = v[c];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
        }
        inc[c] = x;
        if (lane == 31) sh[c * 32 + wid] = x;
    }
    __syncthreads();
    if (wid == 0) {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            int x = sh[c * 32 + lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int y = __shfl_up_sync(0xffffffffu, x, o);
                if (lane >= o) x += y;
            }
            sh[c * 32 + lane] = x;                                  // inclusive over warps
        }
    }
    __syncthreads();
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        v[c] = inc[c] - v[c] + (wid ? sh[c * 32 + wid - 1] : 0);
        tot[c] = sh[c * 32 + 31];
    }
    __syncthreads();
}

__global__ void __launch_bounds__(PLAN_THREADS)
ent2rel_plan_kernel(const int* __restrict__ segptr, int n_rel, int tiles_per_task, int* __restrict__ rel2group,
                    int* __restrict__ group_rel, int* __restrict__ group_tile0, int* __restrict__ task_ptr,
                    int* __restrict__ tile_group, int* __restrict__ task_row0, int* __restrict__ task_row1,
                    int* __restrict__ counts) {
    __shared__ int sh[3 * 32];
    __shared__ int carry[3];
    if (threadIdx.x < 3) carry[threadIdx.x] = 0;
    __syncthreads();
    for (int base = 0; base < n_rel; base += PLAN_THREADS) {
        const int r = base + (int)threadIdx.x;
        const int cnt = r < n_rel ? segptr[r + 1] - segptr[r] : 0;
        const int tiles = (cnt + E2R_TILE - 1) / E2R_TILE;
        int v[3] = {cnt > 0 ? 1 : 0, tiles, (tiles + tiles_per_task - 1) / tiles_per_task};
        int tot[3];
        scan3(v, tot, sh);
        const int g = carry[0] + v[0];
        if (r < n_rel) {
            rel2group[r] = cnt > 0 ? g : -1;
            if (cnt > 0) { group_rel[g] = r; group_tile0[g] = carry[1] + v[1]; task_ptr[g] = carry[2] + v[2]; }
        }
        __syncthreads();
        if (threadIdx.x < 3) carry[threadIdx.x] += tot[threadIdx.x];
        __syncthreads();
    }
    const int n_groups = carry[0];
    if (threadIdx.x == 0) {
        group_tile0[n_groups] = carry[1];
        task_ptr[n_groups] = carry[2];
        counts[0] = n_groups; counts[1] = carry[1]; counts[2] = carry[2];
    }
    __syncthreads();                                                // (global writes of this CTA are visible to it now)
    const int lane = threadIdx.x & 31;
    for (int g = threadIdx.x >> 5; g < n_groups; g += PLAN_THREADS / 32) {
        const int t0 = group_tile0[g], t1 = group_tile0[g + 1];
        for (int t = t0 + lane; t < t1; t += 32) tile_group[t] = g;
        const int r = group_rel[g];
        const int row_end = t0 * E2R_TILE + (segptr[r + 1] - segptr[r]);
        const int z0 = task_ptr[g], z1 = task_ptr[g + 1];
        for (int z = z0 + lane; z < z1; z += 32) {
            const int a = (t0 + (z - z0) * tiles_per_task) * E2R_TILE;
            task_row0[z] = a;
            task_row1[z] = min(a + tiles_per_task * E2R_TILE, row_end);    // pad rows are left out of dW
        }
    }
}

__global__ void ent2rel_positions_kernel(const int* __restrict__ keys, const int* __restrict__ vals, long n, int n_rel,
                                         const int* __restrict__ segptr, const int* __restrict__ rel2group,
                                         const int* __restrict__ group_tile0, long long* __restrict__ pos) {
    const long j = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const int k = keys[j];
    pos[vals[j]] = k < n_rel ? (long long)group_tile0[rel2group[k]] * E2R_TILE + (j - segptr[k]) : 0;
}

// one warp per padded row, grid-stride over the rows of the tiles in use
__global__ void ent2rel_gather_kernel(const float* __restrict__ table, long ldt, long n_table,
                                      const long long* __restrict__ ids, const int* __restrict__ vals,
                                      const int* __restrict__ segptr, const int* __restrict__ group_rel,
                                      const int* __restrict__ group_tile0, const int* __restrict__ tile_group,
                                      const int* __restrict__ counts, int width, float* __restrict__ out, long ldo,
                                      int* __restrict__ err) {
    const int lane = threadIdx.x & 31;
    const long rows = (long)counts[1] * E2R_TILE;
    const long nw = (long)gridDim.x * (blockDim.x >> 5);
    for (long p = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); p < rows; p += nw) {
        const int g = tile_group[p / E2R_TILE];
        const int r = group_rel[g];
        const long local = p - (long)group_tile0[g] * E2R_TILE;
        long row = -1;
        if (local < segptr[r + 1] - segptr[r]) {
            const long src = vals[segptr[r] + local];
            row = ids ? (long)ids[src] : src;
            if (row < 0 || row >= n_table) {
                if (lane == 0) atomicOr(err, 1);
                row = -1;
            }
        }
        float* o = out + p * ldo;
        if (row < 0) {
            for (int c = lane; c < width; c += 32) o[c] = 0.f;
        } else {
            const float* x = table + row * ldt;
            for (int c = lane; c < width; c += 32) o[c] = x[c];
        }
    }
}

bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace
}  // namespace spk

using namespace spk;

extern "C" {

int spk_ent2rel_keys(const int64_t* rel, int64_t stride, int64_t n_src, int32_t reps, int32_t n_rel, int32_t* keys,
                     int32_t* vals, int32_t* err_flag, spk_stream_t stream) {
    if (n_src < 0 || reps < 1 || stride < 1 || n_rel < 1 || n_src * reps >= (1LL << 31)) {
        set_error("ent2rel_keys: bad arguments"); return 1;
    }
    const long n = (long)n_src * reps;
    if (n == 0) return 0;
    ent2rel_keys_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const long long*>(rel), (long)stride, (long)n_src, n, n_rel, keys, vals, err_flag);
    return check_launch("ent2rel_keys");
}

int spk_ent2rel_plan(const int32_t* segptr, int32_t n_rel, int32_t tiles_per_task, int32_t* rel2group,
                     int32_t* group_rel, int32_t* group_tile0, int32_t* task_ptr, int32_t* tile_group,
                     int32_t* task_row0, int32_t* task_row1, int32_t* counts, spk_stream_t stream) {
    if (n_rel < 1 || tiles_per_task < 1) { set_error("ent2rel_plan: bad arguments"); return 1; }
    ent2rel_plan_kernel<<<1, PLAN_THREADS, 0, (cudaStream_t)stream>>>(segptr, n_rel, tiles_per_task, rel2group, group_rel,
                                                                    group_tile0, task_ptr, tile_group, task_row0,
                                                                    task_row1, counts);
    return check_launch("ent2rel_plan");
}

int spk_ent2rel_positions(const int32_t* sorted_keys, const int32_t* sorted_vals, int64_t n_rows, int32_t n_rel,
                          const int32_t* segptr, const int32_t* rel2group, const int32_t* group_tile0, int64_t* pos,
                          spk_stream_t stream) {
    if (n_rows <= 0) return 0;
    ent2rel_positions_kernel<<<(unsigned)((n_rows + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        sorted_keys, sorted_vals, (long)n_rows, n_rel, segptr, rel2group, group_tile0, reinterpret_cast<long long*>(pos));
    return check_launch("ent2rel_positions");
}

int spk_ent2rel_gather(const float* table, int64_t ldt, int64_t n_table, const int64_t* ids, const int32_t* sorted_vals,
                       const int32_t* segptr, const int32_t* group_rel, const int32_t* group_tile0,
                       const int32_t* tile_group, const int32_t* counts, int32_t width, int64_t max_rows, float* out,
                       int64_t ldo, int32_t* err_flag, spk_stream_t stream) {
    if (width < 1 || ldt < width || ldo < width || max_rows % 128) { set_error("ent2rel_gather: bad shape"); return 1; }
    if (max_rows == 0) return 0;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    long blocks = (max_rows + 7) / 8;
    if (blocks > 16L * sms) blocks = 16L * sms;
    ent2rel_gather_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
        table, (long)ldt, (long)n_table, reinterpret_cast<const long long*>(ids), sorted_vals, segptr, group_rel,
        group_tile0, tile_group, counts, width, out, (long)ldo, err_flag);
    return check_launch("ent2rel_gather");
}

int64_t spk_gemm_nn_tc_grouped_workspace_floats(int32_t max_groups, int32_t N, int32_t K) {
    return 2LL * max_groups * N * gemm_tc_ldt(K);
}

int spk_gemm_nn_tc_grouped(const float* A, int64_t lda, int64_t max_rows, const float* W, int64_t rstride, int64_t sn,
                           int64_t sk, int32_t N, int32_t K, const int32_t* group_rel, const int32_t* counts,
                           int32_t max_groups, const int32_t* tile_group, float* C, int64_t ldc, int32_t act,
                           float* workspace, spk_stream_t stream) {
    if (N < 1 || K < 1 || max_groups < 1 || max_rows < 128 || max_rows % 128 || lda < K || ldc < N || (lda & 3) ||
        !al16(A)) {
        set_error("gemm_nn_tc_grouped: A must be 16-byte aligned with lda %% 4 == 0 and lda >= K, max_rows a multiple of 128");
        return 1;
    }
    if (!workspace || !al16(workspace)) { set_error("gemm_nn_tc_grouped: aligned workspace required"); return 1; }
    if (act != 0 && act != 2) { set_error("gemm_nn_tc_grouped: activation %d not supported", act); return 1; }
    return gemm_nn_tc_grouped(A, (long)lda, (long)max_rows, W, (long)rstride, (long)sn, (long)sk, N, K, group_rel, counts,
                              max_groups, tile_group, counts + 1, C, (long)ldc, act, workspace, (cudaStream_t)stream);
}

int64_t spk_gemm_tn_tc_grouped_workspace_floats(int32_t max_tasks, int32_t Ka, int32_t Nb) {
    return gemm_tn_tc_grouped_workspace_floats(max_tasks, Ka, Nb);
}

int spk_gemm_tn_tc_grouped(const float* A, int64_t lda, const float* B, int64_t ldb, int64_t max_rows, int32_t Ka,
                           int32_t Nb, const int32_t* task_row0, const int32_t* task_row1, const int32_t* counts,
                           int32_t max_tasks, const int32_t* rel2group, const int32_t* task_ptr, int32_t n_rel, float* C,
                           float* workspace, spk_stream_t stream) {
    if (Ka < 1 || Nb < 1 || n_rel < 1 || max_tasks < 0 || max_rows < 1 || lda < Ka || ldb < Nb || (lda & 3) || (ldb & 3) ||
        !al16(A) || !al16(B)) {
        set_error("gemm_tn_tc_grouped: operands must be 16-byte aligned with ld %% 4 == 0"); return 1;
    }
    if (max_tasks > 0 && !workspace) { set_error("gemm_tn_tc_grouped: workspace required"); return 1; }
    return gemm_tn_tc_grouped(A, (long)lda, B, (long)ldb, (long)max_rows, Ka, Nb, task_row0, task_row1, counts + 2,
                              max_tasks, rel2group, task_ptr, n_rel, C, workspace, (cudaStream_t)stream);
}

}  // extern "C"
