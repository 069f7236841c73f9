// extern "C" surface of libspkbgat.so (declared in include/spkbgat.h): argument validation and
// translation to the internal launchers. No device allocation, no retained pointers.
#include "../../include/spkbgat.h"
#include "spk_common.cuh"
#include "spk_edge.cuh"
#include "spk_edge_bwd_fused.cuh"
#include "spk_agg.cuh"
#include "spk_gemm.cuh"
#include "spk_graph.cuh"
#include "spk_rowops.cuh"

namespace spk {

static thread_local char g_err[512] = "";
static unsigned long long g_launches = 0;      // kernels launched through this library (bench.py gpu_launches)

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int check_launch(const char* what) {
    const cudaError_t e = cudaGetLastError();
    __atomic_fetch_add(&g_launches, 1ULL, __ATOMIC_RELAXED);
    if (e == cudaSuccess) return 0;
    set_error("%s: CUDA error %d (%s)", what, (int)e, cudaGetErrorString(e));
    return 100 + (int)e;
}

static bool geom_ok(const spk_geom& g, LayerGeom* out, const char* who) {
    if (g.n_heads < 1 || g.n_heads > SPK_MAX_HEADS || g.d_head < 1 || g.d_pad < g.d_head || (g.d_pad & 3) ||
        (g.width & 7) || g.width < g.n_heads * g.d_pad + g.n_heads || g.width > 512) {
        set_error("%s: bad geometry H=%d D=%d Dp=%d Wd=%d", who, g.n_heads, g.d_head, g.d_pad, g.width);
        return false;
    }
    out->H = g.n_heads; out->D = g.d_head; out->Dp4 = g.d_pad / 4;
    out->Dt4 = g.n_heads * g.d_pad / 4; out->Wd4 = g.width / 4;
    return true;
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

static HubTasks hub_of(const spk_hub_tasks& h) {
    HubTasks t;
    t.task_seg = h.task_seg; t.task_beg = h.task_beg; t.task_end = h.task_end;
    t.hub_seg = h.hub_seg; t.hub_task_ptr = h.hub_task_ptr;
    t.partial = h.partial; t.ldpart = h.ldpart;
    t.n_tasks = h.n_tasks; t.n_hubs = h.n_hubs;
    t.hub_thresh = h.n_tasks > 0 ? h.hub_thresh : 0x7fffffff;
    t.task_order = h.n_tasks > 0 ? h.task_order : nullptr;
    return t;
}

// ---- stand-alone SpecialSpmmFunctionFinal -------------------------------------------------------
__global__ void __launch_bounds__(256)
spmm_rowsum_kernel(const int* __restrict__ segptr, const int* __restrict__ perm, const float* __restrict__ w, long ldw,
                   int width, float* __restrict__ out, long ldo, int n_rows) {
    const int lane = threadIdx.x & 31;
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= n_rows) return;
    const int beg = segptr[row], end = segptr[row + 1];
    if (width == 1) {                                    // e_rowsum case (layers.py:150): lanes over edges
        float s = 0.f;
        for (int e = beg + lane; e < end; e += 32) s += w[(long)perm[e] * ldw];
        s = warp_sum(s);
        if (lane == 0) out[(long)row * ldo] = s;
        return;
    }
    for (int c = lane; c < width; c += 32) {
        float s = 0.f;
        for (int e = beg; e < end; ++e) s += w[(long)perm[e] * ldw + c];
        out[(long)row * ldo + c] = s;
    }
}

__global__ void spmm_rowsum_bwd_kernel(const long long* __restrict__ edge_row, const float* __restrict__ g, long ldg,
                                       int width, float* __restrict__ gw, long ldw, long n_edges) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_edges * width) return;
    const long e = i / width; const int c = (int)(i % width);
    gw[e * ldw + c] = g[(long)edge_row[e] * ldg + c];     // layers.py:75
}

}  // namespace spk

using namespace spk;

extern "C" {

int spk_abi_version(void) { return SPK_ABI_VERSION; }
const char* spk_last_error(void) { return g_err; }
int64_t spk_launch_count(void) { return (int64_t)__atomic_load_n(&g_launches, __ATOMIC_RELAXED); }

int spk_edges_concat(const int64_t* edge, int64_t e1, const int64_t* edge_type, const int64_t* nhop, int64_t e2,
                     int32_t* row, int32_t* col, int32_t* t1, int32_t* t2, int64_t n_nodes, int64_t n_rel,
                     int32_t* err_flag, spk_stream_t stream) {
    if (e1 + e2 >= (1LL << 31) || n_nodes >= (1LL << 31)) { set_error("edges_concat: sizes exceed int32"); return 1; }
    if (e2 > 0 && !t2) { set_error("edges_concat: t2 required when 2-hop rows are given"); return 1; }
    return edges_concat(reinterpret_cast<const long long*>(edge), e1, reinterpret_cast<const long long*>(edge_type),
                        reinterpret_cast<const long long*>(nhop), e2, row, col, t1, t2, n_nodes, n_rel, err_flag,
                        (cudaStream_t)stream);
}
int spk_iota_i32(int32_t* v, int64_t n, spk_stream_t stream) { return iota_i32(v, n, (cudaStream_t)stream); }
int64_t spk_sort_workspace_bytes(int64_t n) { return radix_sort_workspace_bytes(n); }
int spk_sort_pairs(int32_t* keys, int32_t* vals, int32_t* keys_tmp, int32_t* vals_tmp, int64_t n, int32_t key_bits,
                   void* workspace, int32_t* result_in_tmp, spk_stream_t stream) {
    if (key_bits < 1 || key_bits > 31) { set_error("sort_pairs: key_bits %d out of range", key_bits); return 1; }
    return radix_sort_pairs(keys, vals, keys_tmp, vals_tmp, n, key_bits, workspace, result_in_tmp, (cudaStream_t)stream);
}
int spk_segment_ptr(const int32_t* sorted_keys, int64_t n, int32_t n_seg, int32_t* ptr, spk_stream_t stream) {
    return segment_ptr(sorted_keys, n, n_seg, ptr, (cudaStream_t)stream);
}
int spk_gather_i32(const int32_t* src, const int32_t* idx, int64_t n, int32_t* out, spk_stream_t stream) {
    return gather_i32(src, idx, n, out, (cudaStream_t)stream);
}
int spk_rel_incidence(const int32_t* t1, const int32_t* t2, int64_t e, int32_t n_rel, int32_t* keys, int32_t* vals,
                      spk_stream_t stream) {
    return rel_incidence(t1, t2, e, n_rel, keys, vals, (cudaStream_t)stream);
}

int spk_gemm_nn(const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc,
                int64_t M, int32_t N, int32_t K, int32_t accumulate, spk_stream_t stream) {
    if (lda < K || ldb < N || ldc < N) { set_error("gemm_nn: leading dimension too small"); return 1; }
    return gemm_nn_simt(A, lda, B, ldb, C, ldc, M, N, K, accumulate, (cudaStream_t)stream);
}
int64_t spk_gemm_tn_workspace_floats(int64_t M, int32_t Ka, int32_t Nb) { return gemm_tn_workspace_floats(M, Ka, Nb); }
int spk_gemm_tn(const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc,
                int64_t M, int32_t Ka, int32_t Nb, int32_t accumulate, float* workspace, spk_stream_t stream) {
    if (lda < Ka || ldb < Nb || ldc < Nb) { set_error("gemm_tn: leading dimension too small"); return 1; }
    if (!workspace) { set_error("gemm_tn: workspace required"); return 1; }
    return gemm_tn_simt(A, lda, B, ldb, C, ldc, M, Ka, Nb, accumulate, workspace, (cudaStream_t)stream);
}

int32_t spk_gemm_nn_tc_supported(const float* A, int64_t lda, int64_t M, int32_t N, int32_t K) {
    return gemm_nn_tc_supported(A, lda, M, N, K);
}
int64_t spk_gemm_tc_workspace_floats(int32_t N, int32_t K) { return 2LL * N * gemm_tc_ldt(K); }
int spk_gemm_nn_tc(const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc,
                   int64_t M, int32_t N, int32_t K, int32_t accumulate, float* workspace, spk_stream_t stream) {
    if (lda < K || ldb < N || ldc < N) { set_error("gemm_nn_tc: leading dimension too small"); return 1; }
    if (!gemm_nn_tc_supported(A, lda, M, N, K)) { set_error("gemm_nn_tc: A must be 16-byte aligned with lda %% 4 == 0"); return 1; }
    if (!workspace || (reinterpret_cast<uintptr_t>(workspace) & 15)) { set_error("gemm_nn_tc: aligned workspace required"); return 1; }
    return gemm_nn_tc(A, lda, B, ldb, C, ldc, M, N, K, accumulate, workspace, (cudaStream_t)stream);
}

int spk_gemm_nn_tc_act(const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc,
                       int64_t M, int32_t N, int32_t K, int32_t accumulate, int32_t act, float* workspace, spk_stream_t stream) {
    if (lda < K || ldb < N || ldc < N) { set_error("gemm_nn_tc_act: leading dimension too small"); return 1; }
    if (!gemm_nn_tc_supported(A, lda, M, N, K)) { set_error("gemm_nn_tc_act: A must be 16-byte aligned with lda %% 4 == 0"); return 1; }
    if (!workspace || (reinterpret_cast<uintptr_t>(workspace) & 15)) { set_error("gemm_nn_tc_act: aligned workspace required"); return 1; }
    if (act < 0 || act > 2) { set_error("gemm_nn_tc_act: unknown activation %d", act); return 1; }
    return gemm_nn_tc(A, lda, B, ldb, C, ldc, M, N, K, accumulate, workspace, (cudaStream_t)stream, act);
}
int spk_elu_inplace(float* x, int64_t ldx, int64_t n_rows, int32_t width, spk_stream_t stream) {
    if (ldx < width) { set_error("elu_inplace: leading dimension too small"); return 1; }
    return launch_elu_inplace(x, ldx, n_rows, width, (cudaStream_t)stream);
}

int32_t spk_gemm_tn_tc_supported(const float* A, int64_t lda, const float* B, int64_t ldb, int64_t M, int32_t Ka, int32_t Nb) {
    return gemm_tn_tc_supported(A, lda, B, ldb, M, Ka, Nb);
}
int64_t spk_gemm_tn_tc_workspace_floats(int64_t M, int32_t Ka, int32_t Nb) { return gemm_tn_tc_workspace_floats(M, Ka, Nb); }
int spk_gemm_tn_tc(const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc,
                   int64_t M, int32_t Ka, int32_t Nb, int32_t accumulate, float* workspace, spk_stream_t stream) {
    if (ldc < Nb) { set_error("gemm_tn_tc: leading dimension too small"); return 1; }
    if (!gemm_tn_tc_supported(A, lda, B, ldb, M, Ka, Nb)) { set_error("gemm_tn_tc: operands must be 16-byte aligned with ld %% 4 == 0"); return 1; }
    if (!workspace) { set_error("gemm_tn_tc: workspace required"); return 1; }
    return gemm_tn_tc(A, lda, B, ldb, C, ldc, M, Ka, Nb, accumulate, workspace, (cudaStream_t)stream);
}

int spk_edge_attn_fwd(const spk_edge_fwd_args* p, spk_stream_t stream) {
    EdgeFwdArgs a;
    if (!geom_ok(p->geom, &a.g, "edge_attn_fwd")) return 1;
    if ((p->ld1 & 3) || (p->ld2 & 3) || (p->ld3 & 3) || p->ld1 < p->geom.width || p->ld2 < p->geom.width ||
        p->ld3 < p->geom.width || !aligned16(p->P1) || !aligned16(p->P2) || !aligned16(p->P3)) {
        set_error("edge_attn_fwd: projected tables must be 16-byte aligned with ld >= width, ld %% 4 == 0");
        return 1;
    }
    a.segptr = p->segptr; a.col = p->col; a.t1 = p->t1; a.t2 = p->t2;
    a.P1 = p->P1; a.ld1 = p->ld1; a.P2 = p->P2; a.ld2 = p->ld2; a.P3 = p->P3; a.ld3 = p->ld3;
    a.mask = p->mask; a.mask_stride = p->mask_stride;
    a.out = p->out; a.ldo = p->ldo; a.den = p->den; a.sw = p->sw; a.nanflag = p->nanflag;
    a.n_rows = p->n_rows; a.alpha = p->alpha; a.apply_elu = p->apply_elu;
    a.elu_rows = p->elu_rows > 0 ? p->elu_rows : 0x7fffffff;
    a.out_vec = (p->geom.d_head % 4 == 0) && (p->ldo % 4 == 0) && aligned16(p->out);
    a.hub = hub_of(p->hub);
    if (a.hub.n_tasks > 0 && (a.hub.ldpart < p->geom.width + 2 * SPK_MAX_HEADS || (a.hub.ldpart & 3) || !aligned16(a.hub.partial))) {
        set_error("edge_attn_fwd: hub partial buffer needs ldpart >= width+8, ldpart %% 4 == 0");
        return 1;
    }
    return launch_edge_fwd(a, (cudaStream_t)stream);
}

int spk_edge_attn_bwd_rows(const spk_edge_bwd_rows_args* p, spk_stream_t stream) {
    EdgeBwdRowsArgs a;
    if (!geom_ok(p->geom, &a.g, "edge_attn_bwd_rows")) return 1;
    if ((p->ld1 & 3) || (p->ld2 & 3) || (p->ld3 & 3) || (p->ldg & 3) || (p->ldd1 & 3) || p->ldg < p->geom.n_heads * p->geom.d_pad ||
        p->ldd1 < p->geom.width || !aligned16(p->P1) || !aligned16(p->P2) || !aligned16(p->P3) || !aligned16(p->G) ||
        !aligned16(p->dP1) || (reinterpret_cast<uintptr_t>(p->rec) & 7)) {
        set_error("edge_attn_bwd_rows: bad leading dimension or alignment");
        return 1;
    }
    a.segptr = p->segptr; a.col = p->col; a.t1 = p->t1; a.t2 = p->t2;
    a.P1 = p->P1; a.ld1 = p->ld1; a.P2 = p->P2; a.ld2 = p->ld2; a.P3 = p->P3; a.ld3 = p->ld3;
    a.mask = p->mask; a.mask_stride = p->mask_stride;
    a.out = p->out; a.dout = p->dout; a.ldo = p->ldo; a.den = p->den;
    a.G = p->G; a.ldg = p->ldg; a.dP1 = p->dP1; a.ldd1 = p->ldd1; a.rec = p->rec;
    a.n_rows = p->n_rows; a.alpha = p->alpha; a.apply_elu = p->apply_elu;
    a.out_vec = (p->geom.d_head % 4 == 0) && (p->ldo % 4 == 0) && aligned16(p->out) && aligned16(p->dout);
    a.hub = hub_of(p->hub);
    if (a.hub.n_tasks > 0 && a.hub.ldpart < 2 * SPK_MAX_HEADS) { set_error("edge_attn_bwd_rows: hub ldpart must be >= 8"); return 1; }
    return launch_edge_bwd_rows(a, (cudaStream_t)stream);
}

int spk_edge_attn_bwd_segments(const spk_seg_gather_args* p, spk_stream_t stream) {
    SegGatherArgs a;
    if (!geom_ok(p->geom, &a.g, "edge_attn_bwd_segments")) return 1;
    if ((p->ldg & 3) || (p->ldout & 3) || p->ldout < p->geom.width || p->ldg < p->geom.n_heads * p->geom.d_pad ||
        !aligned16(p->G) || !aligned16(p->out) || (reinterpret_cast<uintptr_t>(p->rec) & 7)) {
        set_error("edge_attn_bwd_segments: bad leading dimension or alignment");
        return 1;
    }
    a.segptr = p->segptr; a.src = p->src; a.pos = p->pos; a.G = p->G; a.ldg = p->ldg; a.rec = p->rec;
    a.outp = p->out; a.ldout = p->ldout; a.n_seg = p->n_seg; a.prefer_stream = p->flags & 1;
    a.hub = hub_of(p->hub);
    if (a.hub.n_tasks > 0 && (a.hub.ldpart < p->geom.width || (a.hub.ldpart & 3) || !aligned16(a.hub.partial))) {
        set_error("edge_attn_bwd_segments: hub partial buffer needs ldpart >= width");
        return 1;
    }
    return launch_seg_gather(a, (cudaStream_t)stream);
}

static int fused_args_of(const spk_edge_bwd_fused_args* p, BwdFusedArgs& a, const char* who, int dup = 0);

int spk_edge_attn_bwd_fused(const spk_edge_bwd_fused_args* p, spk_stream_t stream) {
    BwdFusedArgs a;
    if (int rc = fused_args_of(p, a, "edge_attn_bwd_fused")) return rc;
    if (reinterpret_cast<uintptr_t>(p->rec) & 7) { set_error("edge_attn_bwd_fused: rec must be 8-byte aligned"); return 1; }
    return launch_edge_bwd_fused(a, (cudaStream_t)stream);
}

int spk_edge_attn_bwd_split(const spk_edge_bwd_split_args* q, spk_stream_t stream) {
    BwdSplitArgs a;
    if (int rc = fused_args_of(&q->base, a.f, "edge_attn_bwd_split", q->dup)) return rc;
    if (q->base.csc_t2 != nullptr) { set_error("edge_attn_bwd_split: graphs with 2-hop edges are not supported"); return 1; }
    if ((q->ldd3 & 3) || q->ldd3 < q->base.geom.width || !aligned16(q->dP3) || !aligned16(q->rec4) ||
        (reinterpret_cast<uintptr_t>(q->dsv) & 3)) {
        set_error("edge_attn_bwd_split: bad leading dimension or alignment");
        return 1;
    }
    a.colptr = a.f.colptr; a.csc_row = a.f.csc_row; a.csc_pos = a.f.csc_pos; a.csc_t1 = a.f.csc_t1;
    a.relptr = q->relptr; a.rel_row = q->rel_row; a.rel_pos = q->rel_pos;
    a.P2 = a.f.P2; a.ld2 = a.f.ld2; a.P3 = a.f.P3; a.ld3 = a.f.ld3; a.mask = a.f.mask; a.mask_stride = a.f.mask_stride;
    a.G = a.f.G; a.ldg = a.f.ldg; a.rowsc = a.f.rowsc; a.rec4 = q->rec4; a.dsv = q->dsv;
    a.dP2 = a.f.dP2; a.ldd2 = a.f.ldd2; a.dP3 = q->dP3; a.ldd3 = q->ldd3;
    a.n_cols = a.f.n_cols; a.n_rel = q->n_rel; a.g = a.f.g; a.alpha = a.f.alpha;
    a.col_hub = a.f.col_hub;
    if (a.f.row_hub.n_tasks > 0 && (a.f.row_hub.partial == nullptr || a.f.row_hub.ldpart < 4)) {
        set_error("edge_attn_bwd_split: row hub partial buffer [n_tasks, >= 4] required");
        return 1;
    }
    a.phases = q->phases == 0 ? 15 : q->phases;
    a.colsum = q->colsum; a.ld_colsum = q->ld_colsum;
    a.rowsum = q->rowsum; a.ld_rowsum = q->ld_rowsum;
    a.G_rel = q->G_rel ? q->G_rel : a.f.G; a.ldg_rel = q->G_rel ? q->ldg_rel : a.f.ldg;
    a.dup = q->dup;
    if ((a.rowsum && a.ld_rowsum < q->base.geom.n_heads) || (q->G_rel && ((q->ldg_rel & 3) || !aligned16(q->G_rel) ||
        q->ldg_rel < q->base.geom.n_heads * q->base.geom.d_pad)) || (a.dup && (a.phases & 1))) {
        set_error("edge_attn_bwd_split: bad rowsum / G_rel / dup arguments");
        return 1;
    }
    if (a.phases < 0 || a.phases > 15 || (a.colsum && a.ld_colsum < q->base.geom.n_heads)) {
        set_error("edge_attn_bwd_split: bad phases / colsum");
        return 1;
    }
    a.rel_hub = hub_of(q->rel_hub);
    if (a.rel_hub.n_tasks > 0 && (a.rel_hub.ldpart < q->base.geom.width || (a.rel_hub.ldpart & 3) || !aligned16(a.rel_hub.partial))) {
        set_error("edge_attn_bwd_split: relation hub partial buffer needs ldpart >= width");
        return 1;
    }
    return launch_edge_bwd_split(a, (cudaStream_t)stream);
}

static int fused_args_of(const spk_edge_bwd_fused_args* p, BwdFusedArgs& a, const char* who, int dup) {
    if (!geom_ok(p->geom, &a.g, who)) return 1;
    const int64_t tab_w = dup ? p->geom.d_pad + 4 : p->geom.width;      // dup: one copy of the vector + the score scalars
    if ((p->ld1 & 3) || (p->ld2 & 3) || (p->ld3 & 3) || (p->ldg & 3) || (p->ldd1 & 3) || (p->ldd2 & 3) ||
        p->ldg < p->geom.n_heads * p->geom.d_pad || p->ldd1 < p->geom.width || p->ldd2 < p->geom.width ||
        (!dup && p->ld1 < p->geom.width) || p->ld2 < tab_w || p->ld3 < tab_w ||
        !aligned16(p->P1) || !aligned16(p->P2) || !aligned16(p->P3) || !aligned16(p->G) || !aligned16(p->dP1) ||
        !aligned16(p->dP2) || !aligned16(p->rowsc)) {
        set_error("%s: bad leading dimension or alignment", who);
        return 1;
    }
    a.rowptr = p->rowptr; a.colptr = p->colptr; a.csc_row = p->csc_row; a.csc_pos = p->csc_pos;
    a.csc_t1 = p->csc_t1; a.csc_t2 = p->csc_t2;
    a.P1 = p->P1; a.ld1 = p->ld1; a.P2 = p->P2; a.ld2 = p->ld2; a.P3 = p->P3; a.ld3 = p->ld3;
    a.mask = p->mask; a.mask_stride = p->mask_stride;
    a.out = p->out; a.dout = p->dout; a.ldo = p->ldo; a.den = p->den; a.sw = p->sw;
    a.G = p->G; a.ldg = p->ldg; a.rowsc = p->rowsc; a.dP1 = p->dP1; a.ldd1 = p->ldd1; a.dP2 = p->dP2; a.ldd2 = p->ldd2;
    a.rec = p->rec; a.n_rows = p->n_rows; a.n_cols = p->n_cols; a.alpha = p->alpha; a.apply_elu = p->apply_elu;
    a.out_vec = (p->geom.d_head % 4 == 0) && (p->ldo % 4 == 0) && aligned16(p->out) && aligned16(p->dout);
    a.row_hub = hub_of(p->row_hub);
    a.col_hub = hub_of(p->col_hub);
    if (a.col_hub.n_tasks > 0 && (a.col_hub.ldpart < p->geom.width || (a.col_hub.ldpart & 3) || !aligned16(a.col_hub.partial))) {
        set_error("%s: hub partial buffer needs ldpart >= width", who);
        return 1;
    }
    return 0;
}

static bool agg_geom_ok(const spk_agg_geom& g, AggGeom* out, const char* who) {
    if (g.n_heads < 1 || g.n_heads > 2 || g.f_chunks < 1 || g.f_chunks > 15 || g.r_chunks < 1 || g.r_chunks > 15 ||
        g.lz != 4 * (2 * g.f_chunks + g.r_chunks)) {
        set_error("%s: bad geometry H=%d f_chunks=%d r_chunks=%d lz=%d", who, g.n_heads, g.f_chunks, g.r_chunks, g.lz);
        return false;
    }
    out->H = g.n_heads; out->Fx4 = g.f_chunks; out->Fr4 = g.r_chunks; out->LZ = g.lz;
    return true;
}

int spk_agg_table(const float* X, int64_t ldx, const float* V, float* T, int64_t ldt, int64_t n_rows, int32_t F,
                  int32_t f_chunks, spk_stream_t stream) {
    if (F < 1 || F > 60 || f_chunks != (F + 3) / 4 || ldt < 4 * f_chunks + 4 || ldx < F || !aligned16(V)) {
        set_error("agg_table: needs 1 <= F <= 60, f_chunks = ceil(F/4), ldt >= 4*f_chunks+4, 16-byte aligned V");
        return 1;
    }
    return launch_agg_table(X, ldx, V, T, ldt, n_rows, F, f_chunks, (cudaStream_t)stream);
}

int spk_agg_fwd(const spk_agg_fwd_args* p, spk_stream_t stream) {
    AggFwdArgs a;
    if (!agg_geom_ok(p->geom, &a.g, "agg_fwd")) return 1;
    const int wx = 4 * a.g.Fx4 + 4, wr = 4 * a.g.Fr4 + 4;
    if ((p->ldxr & 3) || (p->ldxc & 3) || (p->ldr & 3) || (p->ldz & 3) || p->ldxr < wx || p->ldxc < wx || p->ldr < wr ||
        p->ldz < (int64_t)a.g.H * a.g.LZ || !aligned16(p->xrow) || !aligned16(p->xcol) || !aligned16(p->rel) || !aligned16(p->z)) {
        set_error("agg_fwd: tables must be 16-byte aligned with ld %% 4 == 0 and wide enough");
        return 1;
    }
    a.segptr = p->segptr; a.col = p->col; a.t1 = p->t1; a.t2 = p->t2;
    a.Xrow = p->xrow; a.ldxr = p->ldxr; a.Xcol = p->xcol; a.ldxc = p->ldxc; a.Rt = p->rel; a.ldr = p->ldr;
    a.mask = p->mask; a.mask_stride = p->mask_stride;
    a.Z = p->z; a.ldz = p->ldz; a.den = p->den; a.sw = p->sw; a.nanflag = p->nanflag;
    a.n_rows = p->n_rows; a.alpha = p->alpha;
    a.hub = hub_of(p->hub);
    if (a.hub.n_tasks > 0 && (a.hub.ldpart < AGG_LDPART || (a.hub.ldpart & 3) || !aligned16(a.hub.partial))) {
        set_error("agg_fwd: hub partial buffer needs ldpart >= %d, ldpart %% 4 == 0", AGG_LDPART);
        return 1;
    }
    return launch_agg_fwd(a, (cudaStream_t)stream);
}

int spk_agg_bwd_pre(const float* out, const float* dout, int64_t ldo, const float* den, int32_t n_heads, int32_t d_head,
                    int32_t apply_elu, float* dhn, int64_t ldd, float* dden, int64_t n_rows, spk_stream_t stream) {
    if (n_heads < 1 || d_head < 1 || ldo < (int64_t)n_heads * d_head || ldd < (int64_t)n_heads * d_head) {
        set_error("agg_bwd_pre: bad shape");
        return 1;
    }
    return launch_agg_bwd_pre(out, dout, ldo, den, n_heads, d_head, apply_elu, dhn, ldd, dden, n_rows, (cudaStream_t)stream);
}

int spk_agg_bwd_rows(const spk_agg_bwd_args* p, spk_stream_t stream) {
    AggBwdArgs a;
    if (!agg_geom_ok(p->geom, &a.g, "agg_bwd_rows")) return 1;
    const int wx = 4 * a.g.Fx4 + 4, wr = 4 * a.g.Fr4 + 4;
    if ((p->ldxr & 3) || (p->ldxc & 3) || (p->ldr & 3) || (p->ldz & 3) || (p->ldgx & 3) || (p->ldgr & 3) || (p->ldro & 3) ||
        p->ldxr < wx || p->ldxc < wx || p->ldr < wr || p->ldz < (int64_t)a.g.H * a.g.LZ ||
        p->ldgx < (int64_t)a.g.H * 4 * a.g.Fx4 || p->ldgr < (int64_t)a.g.H * 4 * a.g.Fr4 || p->ldro < wx ||
        !aligned16(p->xrow) || !aligned16(p->xcol) || !aligned16(p->rel) || !aligned16(p->dz) || !aligned16(p->gx) ||
        !aligned16(p->gr) || !aligned16(p->rowout) || !aligned16(p->rec) || !p->rowsc || !aligned16(p->rowsc)) {
        set_error("agg_bwd_rows: bad leading dimension or alignment");
        return 1;
    }
    a.segptr = p->segptr; a.col = p->col; a.t1 = p->t1; a.t2 = p->t2;
    a.Xrow = p->xrow; a.ldxr = p->ldxr; a.Xcol = p->xcol; a.ldxc = p->ldxc; a.Rt = p->rel; a.ldr = p->ldr;
    a.mask = p->mask; a.mask_stride = p->mask_stride;
    a.dZ = p->dz; a.ldz = p->ldz; a.den = p->den; a.sw = p->sw; a.dden = p->dden;
    a.Gx = p->gx; a.ldgx = p->ldgx; a.Gr = p->gr; a.ldgr = p->ldgr; a.rowout = p->rowout; a.ldro = p->ldro; a.rowsc = p->rowsc; a.rec = p->rec;
    a.n_rows = p->n_rows; a.alpha = p->alpha;
    a.hub = hub_of(p->hub);
    if (a.hub.n_tasks > 0 && a.hub.ldpart < 8) { set_error("agg_bwd_rows: hub ldpart must be >= 8"); return 1; }
    return launch_agg_bwd_rows(a, (cudaStream_t)stream);
}

int spk_agg_bwd_ctx(const spk_agg_bwd_args* p, spk_stream_t stream) {
    AggBwdArgs a;
    if (!agg_geom_ok(p->geom, &a.g, "agg_bwd_ctx")) return 1;
    const int wx = 4 * a.g.Fx4 + 4;
    if ((p->ldxr & 3) || (p->ldz & 3) || (p->ldgx & 3) || (p->ldgr & 3) || (p->ldro & 3) || p->ldxr < wx ||
        p->ldz < (int64_t)a.g.H * a.g.LZ || p->ldgx < (int64_t)a.g.H * 4 * a.g.Fx4 || p->ldgr < (int64_t)a.g.H * 4 * a.g.Fr4 ||
        p->ldro < wx || !aligned16(p->xrow) || !aligned16(p->dz) || !aligned16(p->gx) || !aligned16(p->gr) ||
        !aligned16(p->rowout) || !p->rowsc || !aligned16(p->rowsc)) {
        set_error("agg_bwd_ctx: bad leading dimension or alignment");
        return 1;
    }
    a.segptr = nullptr; a.col = nullptr; a.t1 = nullptr; a.t2 = nullptr;
    a.Xrow = p->xrow; a.ldxr = p->ldxr; a.Xcol = nullptr; a.ldxc = 0; a.Rt = nullptr; a.ldr = 0;
    a.mask = nullptr; a.mask_stride = 0;
    a.dZ = p->dz; a.ldz = p->ldz; a.den = p->den; a.sw = p->sw; a.dden = p->dden;
    a.Gx = p->gx; a.ldgx = p->ldgx; a.Gr = p->gr; a.ldgr = p->ldgr; a.rowout = p->rowout; a.ldro = p->ldro; a.rowsc = p->rowsc; a.rec = nullptr;
    a.n_rows = p->n_rows; a.alpha = p->alpha;
    return launch_agg_bwd_ctx_split(a, (cudaStream_t)stream);
}

int spk_agg_dx(const float* rowout, int64_t ldro, const float* dxc, int64_t ldc, const float* V, int64_t n_rows, int32_t F,
               int32_t f_chunks, int32_t n_heads, float* dX, int64_t lddx, float* dq, spk_stream_t stream) {
    if (F < 1 || f_chunks != (F + 3) / 4 || n_heads < 1 || n_heads > 2 || ldro < 4 * f_chunks + 4 ||
        ldc < (int64_t)n_heads * 4 * f_chunks + n_heads || lddx < F || !aligned16(V) || !aligned16(dq)) {
        set_error("agg_dx: bad shape or alignment");
        return 1;
    }
    return launch_agg_dx(rowout, ldro, dxc, ldc, V, n_rows, F, f_chunks, n_heads, dX, lddx, dq, (cudaStream_t)stream);
}

int spk_spmm_rowsum_fwd(const int32_t* segptr, const int32_t* perm, const float* w, int64_t ldw, int32_t width,
                        float* out, int64_t ldo, int32_t n_rows, spk_stream_t stream) {
    if (n_rows <= 0) return 0;
    spmm_rowsum_kernel<<<(n_rows + 7) / 8, 256, 0, (cudaStream_t)stream>>>(segptr, perm, w, ldw, width, out, ldo, n_rows);
    return check_launch("spmm_rowsum");
}
int spk_spmm_rowsum_bwd(const int64_t* edge_row, const float* gout, int64_t ldg, int32_t width, float* gw, int64_t ldw,
                        int64_t n_edges, spk_stream_t stream) {
    const long total = n_edges * width;
    if (total <= 0) return 0;
    spmm_rowsum_bwd_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const long long*>(edge_row), gout, ldg, width, gw, ldw, n_edges);
    return check_launch("spmm_rowsum_bwd");
}

int spk_rownorm(const float* x, int64_t ldx, float* y, int64_t ldy, int64_t n_rows, int32_t width, spk_stream_t stream) {
    return rownorm(x, ldx, y, ldy, n_rows, width, (cudaStream_t)stream);
}
int spk_residual_norm_fwd(const float* ew, int64_t lde, const float* x2, int64_t ldx, const float* mask, float* out,
                          int64_t ldo, float* inv_norm, int64_t n_rows, int32_t width, spk_stream_t stream) {
    return residual_norm(ew, lde, x2, ldx, mask, out, ldo, inv_norm, n_rows, width, (cudaStream_t)stream);
}
int spk_residual_norm_bwd(const float* g, int64_t ldg, const float* out, int64_t ldo, const float* mask,
                          const float* inv_norm, float* dew, int64_t lde, float* dx2, int64_t ldx, int64_t n_rows,
                          int32_t width, spk_stream_t stream) {
    return residual_norm_bwd(g, ldg, out, ldo, mask, inv_norm, dew, lde, dx2, ldx, n_rows, width, (cudaStream_t)stream);
}
int spk_mask_from_index(const int64_t* idx, int64_t n_idx, float* mask, int64_t n_rows, int32_t* flag, spk_stream_t stream) {
    return mask_from_index(reinterpret_cast<const long long*>(idx), n_idx, mask, n_rows, flag, (cudaStream_t)stream);
}
static int attn_weights_of(const spk_attn_weights_args* p, AttnWeightsArgs& w, bool bwd) {
    if (!p || p->n_heads < 1 || p->n_heads > 4 || p->F < 1 || p->Rd < 1 || p->D < 1 || (p->mode != 0 && p->mode != 1) ||
        !p->W0 || !p->W1 || (p->mode == 1 && !p->W2)) { set_error("attn_weights: bad arguments"); return 1; }
    for (int h = 0; h < 4; ++h) {
        w.a[h] = h < p->n_heads ? p->a[h] : nullptr; w.a2[h] = h < p->n_heads ? p->a2[h] : nullptr;
        w.da[h] = h < p->n_heads ? p->da[h] : nullptr; w.da2[h] = h < p->n_heads ? p->da2[h] : nullptr;
        if (h < p->n_heads && (!w.a[h] || !w.a2[h] || (bwd && (!w.da[h] || !w.da2[h])))) { set_error("attn_weights: null parameter pointer"); return 1; }
    }
    w.H = p->n_heads; w.F = p->F; w.Rd = p->Rd; w.D = p->D; w.mode = p->mode;
    w.Dp = p->d_pad; w.Dt = p->n_heads * p->d_pad; w.Wd = p->width; w.Fp = p->f_pad; w.LZ = p->lz;
    w.W0 = p->W0; w.ld0 = p->ld0; w.W1 = p->W1; w.ld1 = p->ld1; w.W2 = p->W2;
    if (p->mode == 0 && (p->d_pad < p->D || p->width < w.Dt + p->n_heads || p->ld0 < 2L * p->width || p->ld1 < p->width)) {
        set_error("attn_weights: geometry / leading dimensions too small"); return 1;
    }
    if (p->mode == 1 && (p->f_pad < p->F || p->lz < 2 * p->f_pad + p->Rd || p->n_heads > 2)) {
        set_error("attn_weights: aggregate-then-project geometry"); return 1;
    }
    return 0;
}
int spk_attn_weights_fwd(const spk_attn_weights_args* p, spk_stream_t stream) {
    AttnWeightsArgs w;
    if (int rc = attn_weights_of(p, w, false)) return rc;
    return launch_attn_weights_fwd(w, (cudaStream_t)stream);
}
int spk_attn_weights_bwd(const spk_attn_weights_args* p, spk_stream_t stream) {
    AttnWeightsArgs w;
    if (int rc = attn_weights_of(p, w, true)) return rc;
    return launch_attn_weights_bwd(w, (cudaStream_t)stream);
}

int64_t spk_inner_product_workspace_bytes(void) { return inner_product_workspace_bytes(); }
int spk_inner_product(const float* a, const float* b, int64_t n, void* workspace, float* out, int32_t accumulate,
                      spk_stream_t stream) {
    return inner_product(a, b, n, workspace, out, accumulate, (cudaStream_t)stream);
}

}  // extern "C"
