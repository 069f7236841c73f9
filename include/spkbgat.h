/* libspkbgat -- C ABI of the B200-native SpKBGAT hot path (sm_100a).
 *
 * The reference (ansonb/RECON) has no FFI for this path: its boundary is the Python nn.Module /
 * autograd.Function surface of GAT/layers.py and GAT/models.py. These entry points are what a
 * binding for that path calls instead of the ATen ops listed beside each one. All pointers are raw
 * CUDA device pointers (caller-owned, 16-byte aligned, fp32 / int32 unless stated); the library
 * never allocates or frees device memory and keeps no pointer after a call returns. Every call
 * enqueues on `stream` and returns 0 on success, else a non-zero code with the text available from
 * spk_last_error() (thread-local). See INTEGRATION.md for the ctypes binding the reference-side
 * Python uses.
 *
 * Projected-table row format ("P~ rows", width = spk_geom.width floats, a multiple of 8):
 *     [ n_heads * d_pad projection floats | n_heads score scalars q | zero pad ]
 * d_pad = d_head rounded up to 4; n_heads <= 4 per launch (the host loops over head groups).
 */
#ifndef SPKBGAT_H
#define SPKBGAT_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* spk_stream_t;              /* cudaStream_t */

#define SPK_ABI_VERSION 6
int spk_abi_version(void);
const char* spk_last_error(void);
int64_t spk_launch_count(void);          /* kernels launched through this library so far */

typedef struct {
    int32_t n_heads;   /* H  (1..4) */
    int32_t d_head;    /* D  out_features per head (GAT/layers.py:92 out_features) */
    int32_t d_pad;     /* Dp */
    int32_t width;     /* Wd */
} spk_geom;

/* Segments longer than hub_thresh are processed as chunks (tasks) with partials summed in task
 * order: deterministic handling of power-law hub rows. n_tasks == 0 disables it.
 * task_order (optional, a permutation of [0, n_tasks)): launch slot s runs task task_order[s]; the partial of a task stays
 * at its task index, so the summation order (and every result bit) is independent of it. The relation pass uses it to run
 * the tasks of ALL relations in ascending order of their first aggregation row: the rows gathered by concurrently running
 * tasks then fall into one sliding window that stays L2-resident instead of each relation sweeping the whole table. */
typedef struct {
    const int32_t* task_seg;
    const int32_t* task_beg;
    const int32_t* task_end;
    const int32_t* hub_seg;
    const int32_t* hub_task_ptr;
    float* partial;            /* [n_tasks, ldpart] scratch */
    int64_t ldpart;            /* fwd: width+8 ; bwd_rows: 8 ; seg_gather: width */
    int32_t n_tasks;
    int32_t n_hubs;
    int32_t hub_thresh;
    int32_t reserved;
    const int32_t* task_order; /* [n_tasks] or null */
} spk_hub_tasks;

/* ---- K0: edge construction (replaces the Python/ATen edge prep of GAT/models.py:141-148,
 *      GAT/layers.py:124-127 and the coalesce inside SpecialSpmmFunctionFinal, layers.py:56-58) ---- */
int spk_edges_concat(const int64_t* edge /*[2,E1]*/, int64_t e1, const int64_t* edge_type /*[E1]*/,
                     const int64_t* nhop /*[E2,4] = s,r1,r2,t*/, int64_t e2,
                     int32_t* row, int32_t* col, int32_t* t1, int32_t* t2 /*null if e2==0*/,
                     int64_t n_nodes, int64_t n_rel, int32_t* err_flag, spk_stream_t stream);
/* HOST pointers: dst[i] = (int32) src[i * stride], range-checked against [lo, hi) by n_threads host threads (0 = all):
 * packs the reference API's int64 index tensors into a pinned int32 staging buffer so that half the bytes cross PCIe;
 * returns 5 if a value is out of range. Used by recon_b200.KGraph for host-resident edge tensors. */
int spk_pack_index_host(const int64_t* src, int64_t n, int64_t stride, int64_t lo, int64_t hi, int32_t* dst, int32_t n_threads);
int spk_iota_i32(int32_t* v, int64_t n, spk_stream_t stream);
int64_t spk_sort_workspace_bytes(int64_t n);
/* stable LSD radix sort of (key,value) pairs on the low key_bits bits; result_in_tmp tells which buffers hold it */
int spk_sort_pairs(int32_t* keys, int32_t* vals, int32_t* keys_tmp, int32_t* vals_tmp, int64_t n, int32_t key_bits,
                   void* workspace, int32_t* result_in_tmp, spk_stream_t stream);
int spk_segment_ptr(const int32_t* sorted_keys, int64_t n, int32_t n_seg, int32_t* ptr /*[n_seg+1]*/, spk_stream_t stream);
int spk_gather_i32(const int32_t* src, const int32_t* idx, int64_t n, int32_t* out, spk_stream_t stream);
int spk_rel_incidence(const int32_t* t1, const int32_t* t2, int64_t e, int32_t n_rel, int32_t* keys, int32_t* vals,
                      spk_stream_t stream);

/* ---- K1/K5: dense products (replace a.mm(edge_h) layers.py:137, relation_embed.mm(W) models.py:77,
 *      entity_embeddings.mm(W_entities) models.py:175 and their autograd) ---- */
int spk_gemm_nn(const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc,
                int64_t M, int32_t N, int32_t K, int32_t accumulate, spk_stream_t stream);
int64_t spk_gemm_tn_workspace_floats(int64_t M, int32_t Ka, int32_t Nb);
/* C[Ka,Nb] (+)= A[M,Ka]^T * B[M,Nb], deterministic split over M */
int spk_gemm_tn(const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc,
                int64_t M, int32_t Ka, int32_t Nb, int32_t accumulate, float* workspace, spk_stream_t stream);

/* Same product on the tcgen05 tensor cores: 3xTF32 error-compensated (fp32-accurate), TMA-fed, TMEM accumulators.
 * Needs A 16-byte aligned with lda % 4 == 0 (spk_gemm_nn_tc_supported) and 2*N*roundup(K,4) floats of workspace. */
int32_t spk_gemm_nn_tc_supported(const float* A, int64_t lda, int64_t M, int32_t N, int32_t K);
int64_t spk_gemm_tc_workspace_floats(int32_t N, int32_t K);
int spk_gemm_nn_tc(const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc,
                   int64_t M, int32_t N, int32_t K, int32_t accumulate, float* workspace, spk_stream_t stream);

/* Same, with an epilogue on the final value: act = 0 none, 1 = ELU (F.elu at GAT/layers.py:175 / models.py:86),
 * 2 = tanh (GAT_sep_space/models.py:316-320; the tanhf of spk_tanh_fwd, bit-equal to the product followed by it). */
int spk_gemm_nn_tc_act(const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc,
                       int64_t M, int32_t N, int32_t K, int32_t accumulate, int32_t act, float* workspace,
                       spk_stream_t stream);
int spk_elu_inplace(float* x, int64_t ldx, int64_t n_rows, int32_t width, spk_stream_t stream);

/* C[Ka,Nb] (+)= A[M,Ka]^T * B[M,Nb] on tcgen05 (MN-major operands, both split hi/lo in shared memory),
 * one CTA per (tile, m-split), partials added in split order. */
int32_t spk_gemm_tn_tc_supported(const float* A, int64_t lda, const float* B, int64_t ldb, int64_t M, int32_t Ka, int32_t Nb);
int64_t spk_gemm_tn_tc_workspace_floats(int64_t M, int32_t Ka, int32_t Nb);
int spk_gemm_tn_tc(const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc,
                   int64_t M, int32_t Ka, int32_t Nb, int32_t accumulate, float* workspace, spk_stream_t stream);

/* ---- K2: fused attention forward (replaces SpGraphAttentionLayer.forward layers.py:124-175 for all
 *      heads of a group, incl. both SpecialSpmmFinal calls, the divide and the ELU) ---- */
typedef struct {
    const int32_t* segptr; const int32_t* col; const int32_t* t1; const int32_t* t2;
    const float* P1; int64_t ld1;
    const float* P2; int64_t ld2;
    const float* P3; int64_t ld3;
    const float* mask; int64_t mask_stride;      /* [H][E] CSR-order dropout multipliers or null */
    float* out; int64_t ldo;                     /* [n_rows, H*D] */
    float* den; float* sw;                       /* [n_rows, H] */
    int32_t* nanflag;                            /* sticky: set to 1 where the reference would assert (layers.py:147,167,172) */
    int32_t n_rows; int32_t apply_elu; float alpha;
    int32_t elu_rows;                            /* > 0 with apply_elu: ELU only on rows < elu_rows (0: all rows) */
    spk_geom geom;
    spk_hub_tasks hub;
} spk_edge_fwd_args;
int spk_edge_attn_fwd(const spk_edge_fwd_args* args, spk_stream_t stream);

/* ---- K3: backward over aggregation rows (autograd of layers.py:129-175, SpecialSpmmFunctionFinal.backward 67-79) ---- */
typedef struct {
    const int32_t* segptr; const int32_t* col; const int32_t* t1; const int32_t* t2;
    const float* P1; int64_t ld1;
    const float* P2; int64_t ld2;
    const float* P3; int64_t ld3;
    const float* mask; int64_t mask_stride;
    const float* out; const float* dout; int64_t ldo;
    const float* den;
    float* G; int64_t ldg;                       /* [n_rows, ldg] dnum */
    float* dP1; int64_t ldd1;                    /* [n_rows, width] */
    float* rec;                                  /* [E, 2H] (w, ds) */
    int32_t n_rows; int32_t apply_elu; float alpha; int32_t reserved;
    spk_geom geom;
    spk_hub_tasks hub;
} spk_edge_bwd_rows_args;
int spk_edge_attn_bwd_rows(const spk_edge_bwd_rows_args* args, spk_stream_t stream);

/* ---- K4: backward segmented gather-sum, keyed on edge[1] (dP2~) or on relation id (dP3~) ---- */
typedef struct {
    const int32_t* segptr; const int32_t* src; const int32_t* pos;
    const float* G; int64_t ldg;
    const float* rec;
    float* out; int64_t ldout;                   /* [n_seg, width] */
    int32_t n_seg;
    int32_t flags;                               /* bit 0: many short segments -> 32-segments-per-warp streaming kernel */
    spk_geom geom;
    spk_hub_tasks hub;
} spk_seg_gather_args;
int spk_edge_attn_bwd_segments(const spk_seg_gather_args* args, spk_stream_t stream);

/* ---- K3'/K4': column-major fused backward of a projected layer group. Same outputs as spk_edge_attn_bwd_rows followed by
 *      spk_edge_attn_bwd_segments over the CSC (G, rec, dP1~, dP2~), but every edge is visited once, from its gathered
 *      node: a node pass (dnum, per-row scalars), one pass over the columns (P2~[j] in registers, gathers dnum[i] and the
 *      cache-resident P3~[k], writes the (w, ds) records and dP2~[j]) and a row-sum pass over the records. The relation
 *      pass (dP3~) stays spk_edge_attn_bwd_segments. csc_t1 / csc_t2 are t1 / t2 gathered into CSC order. ---- */
typedef struct {
    const int32_t* rowptr;
    const int32_t* colptr; const int32_t* csc_row; const int32_t* csc_pos; const int32_t* csc_t1; const int32_t* csc_t2;
    const float* P1; int64_t ld1;
    const float* P2; int64_t ld2;
    const float* P3; int64_t ld3;
    const float* mask; int64_t mask_stride;      /* [H][E] CSR-order dropout multipliers or null */
    const float* out; const float* dout; int64_t ldo;
    const float* den; const float* sw;           /* [n_rows, H] from spk_edge_attn_fwd */
    float* G; int64_t ldg;                       /* [n_rows, ldg] dnum */
    float* rowsc;                                /* [n_rows, H, 4] scratch */
    float* dP1; int64_t ldd1;                    /* [n_rows, width] */
    float* dP2; int64_t ldd2;                    /* [n_cols, width] */
    float* rec;                                  /* [E, 2H] (w, ds) in CSR order */
    int32_t n_rows; int32_t n_cols; int32_t apply_elu; float alpha;
    spk_geom geom;
    spk_hub_tasks row_hub;                       /* hub rows (no partial buffer needed) */
    spk_hub_tasks col_hub;                       /* hub columns; partial [n_tasks, ldpart >= width] */
} spk_edge_bwd_fused_args;
int spk_edge_attn_bwd_fused(const spk_edge_bwd_fused_args* args, spk_stream_t stream);

/* ---- K3"/K4": the same backward for graphs without 2-hop edges, with the per-edge dot t = dnum_i . m_e split between the
 *      column pass (dnum_i . P2[j], P2~[j] in registers) and the relation pass (dnum_i . P3[k], P3~[k] in registers), the two
 *      passes that gather dnum_i anyway: no projected row is gathered per edge at all. Computes G, dP1~, dP2~ AND dP3~.
 *      rec4 [E, H, 4] and dsv [E, H] are scratch in CSR order.
 *      `phases` (0 = all) selects what one call launches, so that a multi-GPU caller can start the reduce-scatter of the
 *      partial dP2~ (SURVEY.md 8e) right after the column pass and overlap it with the rest:
 *        1 = node pass (G, rowsc, dP1~ without its q slot)
 *        2 = column pass (rec4, dP2~ without its q slot)
 *        4 = relation pass (dsv, dP3~) + row sums of ds (q slot of dP1~)
 *        8 = column sums of ds: into the q slot of dP2~, or, when `colsum` is given, into colsum[col * ld_colsum + h]
 *      Phases must run in the order 1, 2, 4, 8 on one stream (any grouping: 3 then 12, or one call with 0 = 15). ---- */
typedef struct {
    spk_edge_bwd_fused_args base;                /* csc_t2 must be null; rec unused; col_hub as there; row_hub.partial [n_tasks, >= 4] */
    const int32_t* relptr; const int32_t* rel_row; const int32_t* rel_pos;
    float* rec4; float* dsv;
    float* dP3; int64_t ldd3;                    /* [n_rel, width] */
    int32_t n_rel; int32_t phases;
    spk_hub_tasks rel_hub;                       /* relation segments as tasks; partial [n_tasks, ldpart >= width] */
    float* colsum; int64_t ld_colsum;            /* optional [n_cols, ld_colsum >= n_heads] destination of phase 8 */
    float* rowsum; int64_t ld_rowsum;            /* optional [n_rows, ld_rowsum >= n_heads] destination of the row sums (phase 4) */
    const float* G_rel; int64_t ldg_rel;         /* rows the relation pass gathers (null: base.G) */
    int32_t dup; int32_t reserved;               /* 1: aggregate-then-project tables (see below) */
} spk_edge_bwd_split_args;
/* dup = 1 runs the same column / relation passes for the aggregate-then-project layer (spk_agg_*): base.P2 = X~ and base.P3 =
 * Rel~ (rows [v (d_pad floats) | n_heads score scalars | pad], ld >= d_pad + 4: the SAME input row serves every head), base.G =
 * Gx and G_rel = Gr ([n_rows, n_heads * d_pad], from spk_agg_bwd_ctx), geom.d_head = the input width; phases 2 | 4 | 8 only
 * (spk_agg_bwd_ctx is the node pass). The per-edge dot t = c + Yb . x_j + Yc . r_k is then split over the two passes that gather
 * Gx / Gr anyway, and the row-major regather of X~[j] (spk_agg_bwd_rows' stream kernel) is not needed. */
int spk_edge_attn_bwd_split(const spk_edge_bwd_split_args* args, spk_stream_t stream);

/* ---- K2'/K3': "aggregate-then-project" variant for layer groups whose input is narrower than their projection
 *      (layer 1: in=50, nrela=50 against heads*out=200). Same reference lines as K2/K3 (GAT/layers.py:124-175 and
 *      their autograd); the sum over a row's edges is linear in [x_i | x_j | r_k], so the edges gather the INPUT
 *      rows and a.mm(.) (layers.py:137) is applied once per row to the aggregate by spk_gemm_nn_tc_act:
 *          Zn_h[i] = [ (sum w) x_i | sum w x_j | sum w r_k ] / sum ee      out_h = ELU(Zn_h . a_h^T)
 *      Table rows ("X~", "Rel~"), built by spk_agg_table: [ x | 0-pad to 4*chunks | 4 score scalars | 0-pad ];
 *      X~ scalars = (q2_0, q2_1, q1_0, q1_1), Rel~ scalars = (q3_0, q3_1, 0, 0), q* = x . (A*^T a_2^T).
 *      Needs n_heads <= 2, f_chunks <= 15, r_chunks <= 15. ---- */
typedef struct {
    int32_t n_heads;   /* 1..2 */
    int32_t f_chunks;  /* ceil(in_features / 4) */
    int32_t r_chunks;  /* ceil(nrela_dim / 4) */
    int32_t lz;        /* 4 * (2*f_chunks + r_chunks): floats of Zn per head */
} spk_agg_geom;
/* T[i, :ldt] = [ X[i, :F] | 0 | X[i] . V[:, 0..3] | 0 ],  V is [F, 4] contiguous, ldt >= 4*f_chunks + 4 */
int spk_agg_table(const float* X, int64_t ldx, const float* V, float* T, int64_t ldt, int64_t n_rows,
                  int32_t F, int32_t f_chunks, spk_stream_t stream);
typedef struct {
    const int32_t* segptr; const int32_t* col; const int32_t* t1; const int32_t* t2;
    const float* xrow; int64_t ldxr;             /* X~ of the aggregation rows */
    const float* xcol; int64_t ldxc;             /* X~ of the gathered nodes */
    const float* rel; int64_t ldr;               /* Rel~ */
    const float* mask; int64_t mask_stride;      /* [H][E] CSR-order dropout multipliers or null */
    float* z; int64_t ldz;                       /* [n_rows, H*lz] */
    float* den; float* sw;                       /* [n_rows, H] */
    int32_t* nanflag;
    int32_t n_rows; float alpha;
    spk_agg_geom geom;
    spk_hub_tasks hub;                           /* partial: [n_tasks, 264] */
} spk_agg_fwd_args;
int spk_agg_fwd(const spk_agg_fwd_args* args, spk_stream_t stream);
/* dhn = dout * ELU'(hn) (from the saved output), dden_h = -(dhn_h . hn_h) / den_h */
int spk_agg_bwd_pre(const float* out, const float* dout, int64_t ldo, const float* den, int32_t n_heads, int32_t d_head,
                    int32_t apply_elu, float* dhn, int64_t ldd, float* dden, int64_t n_rows, spk_stream_t stream);
typedef struct {
    const int32_t* segptr; const int32_t* col; const int32_t* t1; const int32_t* t2;
    const float* xrow; int64_t ldxr; const float* xcol; int64_t ldxc; const float* rel; int64_t ldr;
    const float* mask; int64_t mask_stride;
    const float* dz; int64_t ldz;                /* [n_rows, H*lz] gradient w.r.t. Zn (= dhn . a_h) */
    const float* den; const float* sw; const float* dden;
    float* gx; int64_t ldgx;                     /* [n_rows, H*4*f_chunks] rows gathered by the column pass (K4) */
    float* gr; int64_t ldgr;                     /* [n_rows, H*4*r_chunks] rows gathered by the relation pass (K4) */
    float* rowout; int64_t ldro;                 /* [n_rows, 4*f_chunks+4]: dX row part | dq1_0 dq1_1 0 0 */
    float* rowsc;                                /* [n_rows, 8] scratch (per-row scalars between the two kernels) */
    float* rec;                                  /* [E, 2H] (w, ds) */
    int32_t n_rows; float alpha;
    spk_agg_geom geom;
    spk_hub_tasks hub;                           /* partial: [n_tasks, 8] */
} spk_agg_bwd_args;
int spk_agg_bwd_rows(const spk_agg_bwd_args* args, spk_stream_t stream);
/* row-context kernel alone (Gx, Gr, rowout, rowsc as [n_rows, n_heads, 4] = (q1, c, dden, 0)); rec / mask / hub unused */
int spk_agg_bwd_ctx(const spk_agg_bwd_args* args, spk_stream_t stream);
/* dX[i,f] = rowout[i,f] + sum_h dxc[i, h*4*f_chunks + f] + sum_c dq[i,c] V[f,c]; also emits dq [n,4] = (dq2_0,dq2_1,dq1_0,dq1_1).
 * dxc is the K4 column-pass output with geometry (H, d_head = d_pad = 4*f_chunks). */
int spk_agg_dx(const float* rowout, int64_t ldro, const float* dxc, int64_t ldc, const float* V, int64_t n_rows,
               int32_t F, int32_t f_chunks, int32_t n_heads, float* dX, int64_t lddx, float* dq, spk_stream_t stream);

/* ---- stand-alone SpecialSpmmFunctionFinal (layers.py:51-79): out[i,:] = sum_{e in seg i} w[perm[e],:] ---- */
int spk_spmm_rowsum_fwd(const int32_t* segptr, const int32_t* perm, const float* w, int64_t ldw, int32_t width,
                        float* out, int64_t ldo, int32_t n_rows, spk_stream_t stream);
int spk_spmm_rowsum_bwd(const int64_t* edge_row /*[E] original order*/, const float* gout, int64_t ldg, int32_t width,
                        float* gw, int64_t ldw, int64_t n_edges, spk_stream_t stream);

/* ---- K6: row-wise wrappers (models.py:160-161, 167-179) ---- */
int spk_rownorm(const float* x, int64_t ldx, float* y, int64_t ldy, int64_t n_rows, int32_t width, spk_stream_t stream);
int spk_residual_norm_fwd(const float* ew, int64_t lde, const float* x2, int64_t ldx, const float* mask,
                          float* out, int64_t ldo, float* inv_norm, int64_t n_rows, int32_t width, spk_stream_t stream);
int spk_residual_norm_bwd(const float* g, int64_t ldg, const float* out, int64_t ldo, const float* mask,
                          const float* inv_norm, float* dew, int64_t lde, float* dx2, int64_t ldx,
                          int64_t n_rows, int32_t width, spk_stream_t stream);
/* idx may hold negative (from-the-end) indices; one outside [-n_rows, n_rows) ORs 2 into *flag (nullable): the same sticky
 * flag word as `nanflag`, read back once per forward (1: the reference's isnan assertion, 2: its IndexError) */
int spk_mask_from_index(const int64_t* idx, int64_t n_idx, float* mask, int64_t n_rows, int32_t* flag, spk_stream_t stream);
/* out[0] (+)= <a, b> over n contiguous floats (16-byte aligned), deterministic (fixed chunking, fp64 across threads):
 * the linear probe loss <out_entity, G_e> + <out_relation, G_r> of SURVEY.md 8d (the reference's step writes it as
 * (out * G).sum()). workspace: spk_inner_product_workspace_bytes() bytes of device memory. */
/* ---- extended weight matrices from the reference-shaped attention parameters a_h [D, 2F+Rd], a_2,h [1, D]
 *      (GAT/layers.py:100-105), and the gradients back to them: replaces the slice assignments / a.t() / (a^T * a_2).sum()
 *      glue and its autograd.
 *   mode 0 (projected tables, spk_geom):   W0 = Wn [F, ld0 >= 2*width], W1 = Wr [Rd, ld1 >= width]
 *   mode 1 (aggregate-then-project):       W0 = Wa [n_heads, lz, D] (dense), W1 = V [F, 4], W2 = V3 [Rd, 4]
 * spk_attn_weights_fwd zero-fills the outputs and scatters a^T and a^T a_2^T; spk_attn_weights_bwd reads the gradients of
 * the same buffers from W0 / W1 / W2 and writes da[h] (like a[h]) and da2[h] ([D]). n_heads <= 4. ---- */
typedef struct {
    const float* a[4]; const float* a2[4];
    float* da[4]; float* da2[4];
    int32_t n_heads, F, Rd, D;
    int32_t mode; int32_t d_pad, width;         /* mode 0: spk_geom.d_pad / width */
    int32_t f_pad, lz;                           /* mode 1: F rounded up to 4; rows per head of Wa (2 * f_pad + Rd rounded up to 4) */
    int32_t reserved;
    float* W0; int64_t ld0;
    float* W1; int64_t ld1;
    float* W2;
} spk_attn_weights_args;
int spk_attn_weights_fwd(const spk_attn_weights_args* args, spk_stream_t stream);
int spk_attn_weights_bwd(const spk_attn_weights_args* args, spk_stream_t stream);

int64_t spk_inner_product_workspace_bytes(void);
int spk_inner_product(const float* a, const float* b, int64_t n, void* workspace, float* out, int32_t accumulate,
                      spk_stream_t stream);

/* ---- N1 (SURVEY.md 8f): the training step right after the hot path ----
 * batch_gat_loss (GAT/main.py:344-376): `triples` int64 [T,3] = (head, relation, tail) rows, the first n_pos positive,
 * the remaining T - n_pos = 2*ratio*n_pos corrupted (negative k pairs with positive k mod n_pos, main.py:351);
 * x = ent[h] + rel[r] - ent[t], L1 norm, nn.MarginRankingLoss(margin) with y = -1 (main.py:367-372,451),
 * mean != 0: mean over the pairs (the reference's reduction), else sum. Outputs: loss[1]; saved for backward:
 * sgn uint32 [T, ceil(width/4)] (int8 sign(x) packed by 4) and coef float [T] (d loss / d norm of every triple).
 * norm float [T] and partial double [spk_margin_loss_partials(n_pos)] are scratch. Out-of-range ids set *err_flag. */
int64_t spk_margin_loss_partials(int64_t n_pos);
int spk_margin_loss_fwd(const int64_t* triples, int64_t n_triples, int64_t n_pos,
                        const float* ent, int64_t lde, int64_t n_ent, const float* rel, int64_t ldr, int64_t n_rel,
                        int32_t width, float margin, int32_t mean,
                        float* norm, uint32_t* sgn, float* coef, double* partial, float* loss,
                        int32_t* err_flag, spk_stream_t stream);
/* incidence lists for the backward: entity keys (2 per triple, value = 2*t + is_tail) and relation keys (value = t);
 * sorted with spk_sort_pairs and cut into segments with spk_segment_ptr by the caller. */
int spk_triple_incidence(const int64_t* triples, int64_t n_triples, int64_t n_ent, int64_t n_rel,
                         int32_t* ent_keys /*[2T]*/, int32_t* ent_vals, int32_t* rel_keys /*[T]*/, int32_t* rel_vals,
                         int32_t* err_flag, spk_stream_t stream);
/* Backward of batch_gat_loss w.r.t. entity_embed (mode 0) or relation_embed (mode 1): replaces autograd's
 * index_put_(accumulate) scatter. out[seg,:] = gscale[0] * sum over the segment's incidences, in list order, of
 * (+-) coef[t] * sign(x_t)  (- for tails); rows without incidences are written as zeros (dense gradient, the form
 * SpKBGATModified's backward consumes). Deterministic; hub segments through task partials [n_tasks, ldpart >= 4*ceil(width/4)]. */
typedef struct {
    const int32_t* segptr; const int32_t* inc;     /* [n_seg+1], sorted incidence values */
    const float* coef; const uint32_t* sgn;        /* from spk_margin_loss_fwd */
    const float* gscale;                           /* [1] upstream gradient of the scalar loss (device) */
    float* out; int64_t ldo;                       /* [n_seg, width] */
    int32_t n_seg; int32_t width; int32_t mode; int32_t reserved;
    spk_hub_tasks hub;
} spk_loss_bwd_args;
int spk_margin_loss_bwd(const spk_loss_bwd_args* args, spk_stream_t stream);
/* optimizer.step() of torch.optim.SGD(lr) (main.py:445-446,524): param[i] -= lr * grad[i], up to 16 tensors per launch */
typedef struct {
    float* param[16]; const float* grad[16]; int64_t numel[16];
    int32_t count; float lr;
} spk_sgd_args;
int spk_sgd_step(const spk_sgd_args* args, spk_stream_t stream);

/* ---- N2 (SURVEY.md 8f): the embedding wire format the downstream half of RECON reads. HOST pointers, no GPU work. ----
 * spk_export_json writes byte-for-byte what save_embed (GAT/main.py:406-413) writes with
 * json.dump({idx: row.tolist()}, f, indent=4, cls=CustomEncoder): keys "0".."rows-1", one float per line formatted like
 * Python's repr of the float32 widened to double; rows are formatted by n_threads host threads (0 = all cores).
 * spk_export_bin writes the side-car: 64-byte header {"SPKEMB01", int64 rows, int64 width, int64 dtype = 0 (fp32 LE)}
 * followed by rows*width fp32 row-major. */
int spk_export_json(const float* host_rows, int64_t rows, int64_t width, int64_t ld, const char* path, int32_t n_threads);
int spk_export_bin(const float* host_rows, int64_t rows, int64_t width, int64_t ld, const char* path);
/* Reader of that JSON text (what the consumer's json.load does, train.py:103-104, without a Python object per float):
 * spk_import_json_shape returns the number of keys and the length of the first list; spk_import_json parses
 * {"<i>": [numbers], ...} with n_threads host threads (0 = all cores) into out[i, :width] (fp32, row stride ld). */
int spk_import_json_shape(const char* path, int64_t* rows, int64_t* width);
int spk_import_json(const char* path, float* out, int64_t rows, int64_t width, int64_t ld, int32_t n_threads);

/* ---- N3 (SURVEY.md 8f): Corpus.get_iteration_triples_batch (GAT/create_batch.py:262-351) on the device ----
 * spk_triple_keys: key[i] = (h*R + r)*N + t of triples int64 [M,3]; pass the triples in (h, r, t) lexicographic order to
 * get the sorted membership array that stands in for valid_triples_dict (create_batch.py:82-83).
 * spk_corrupt_triples: out_indices int64 [(2*ratio+1)*P, 3], out_values float [(2*ratio+1)*P]: the P positives, then
 * 2*ratio tiled copies of which [0, P*(ratio/2)) get a corrupted head, the next P*(ratio/2) a corrupted tail, rows from
 * P*ratio on a corrupted relation (value -1; see the layout in csrc/spk_sampler.cu). init_entities / init_relations
 * (int64 [P*ratio], may be null) are the first candidates, exactly the reference's random_entities / random_relations;
 * a candidate that makes a valid triple is redrawn from a counter-based generator keyed on (seed, slot, attempt). */
int spk_triple_keys(const int64_t* triples, int64_t n_triples, int64_t n_ent, int64_t n_rel, int64_t* keys,
                    int32_t* err_flag, spk_stream_t stream);
int spk_corrupt_triples(const int64_t* positives, int64_t n_pos, int32_t ratio, const int64_t* valid_keys, int64_t n_valid,
                        int64_t n_ent, int64_t n_rel, const int64_t* init_entities, const int64_t* init_relations,
                        uint64_t seed, int64_t* out_indices, float* out_values, spk_stream_t stream);

/* ---- K0b (SURVEY.md 8 a-1, 8b "spk_nhop_build"): batch adjacency + 2-hop path rows of a batch of source entities, bit-exact
 * (values and order) with Corpus.get_batch_adj_data / bfs / get_batch_nhop_neighbors_all (GAT/create_batch.py:391-436,
 * 788-895). The triple graph is the distinct-neighbour adjacency in the reference's insertion order (int32 device arrays):
 *   uptr [n_nodes+1]  first pair of every head         ut  [n_pairs]  tail of the pair (first-seen order per head)
 *   ur0  [n_pairs]    first relation of the pair       ugs / uge [n_pairs]  range of its parallel relations in rs
 *   rs   [n_triples]  relation ids grouped by (head, tail), file order inside a group
 * Sizes are data dependent: every buffer (scratch and results) is obtained from `alloc` (the caller's allocator, e.g.
 * PyTorch's; must return 16-byte aligned device memory that stays valid until the caller releases it); the call
 * synchronises the stream to read the sizes back. Results: adj_idx int64 [2, e1] = [trgts; srcs], adj_val int64 [e1],
 * nhop int32 [e2, 4] rows [s, r(s->m)[0], r(m->t)[0], t]. flags: bit 0 = partial_2hop (create_batch.py:883-884: the first
 * path of every source only), bit 1 = adjacency only (no 2-hop rows). */
typedef void* (*spk_alloc_fn)(void* ctx, int64_t bytes);
typedef struct {
    const int32_t* uptr; const int32_t* ut; const int32_t* ur0; const int32_t* ugs; const int32_t* uge; const int32_t* rs;
    int32_t n_nodes; int32_t n_pairs; int32_t n_triples; int32_t reserved;
} spk_triple_graph;
typedef struct {
    int64_t* adj_idx; int64_t* adj_val; int32_t* nhop;
    int64_t e1; int64_t e2;
} spk_nhop_result;
int spk_nhop_build(const spk_triple_graph* graph, const int64_t* sources, int64_t n_sources, int32_t flags,
                   spk_alloc_fn alloc, void* alloc_ctx, spk_nhop_result* result, spk_stream_t stream);

/* ---- N4 (SURVEY.md 8f): ConvKB scoring of the hot path's output embeddings ----
 * Reference: ConvKB.forward GAT/layers.py:31-48 (live path fc2(LeakyReLU(fc1([h|r|t])))), SpKBGATConvOnly.forward /
 * batch_test GAT/models.py:294-304, tanh(e . W_ent2rel[r]) GAT_sep_space/models.py:316-320, the all-relations ranking of
 * GAT/create_batch.py:1367-1393. The dense products go through spk_gemm_nn_tc / spk_gemm_tn_tc.
 * spk_gather_concat: out[b, p*D:(p+1)*D] = src[p][row, :D], row = idx[p] ? idx[p][b*stride[p]] : b, for p < n_pieces <= 3
 *                    (the [h|r|t] concatenation from an int64 [B,3] triple tensor: idx = triples+p, stride = 3);
 *                    an index outside [0, rows[p]) sets *err_flag (and reads row 0).
 * spk_mlp_head_fwd:  out[b] = b2 + sum_d w2[d] * lrelu(H1[b,d] + b1[d])            (fc1 bias + LeakyReLU + fc2)
 * spk_mlp_head_bwd:  dH1[b,d] = dout[b] * w2[d] * lrelu'(pre), act[b,d] = lrelu(pre)
 * spk_tanh_fwd / _bwd: x = tanh(x) in place;  dpre = dout * (1 - y^2)
 * spk_rank_scores:   out[i,r] = b2 + sum_d w2[d] * lrelu(U[i,d] + Bt[r,d]), the re-associated fc1: U = A[h] + C[t] + b1 per
 *                    test pair, Bt = Rel . W1b^T per relation; D <= 512. */
int spk_gather_concat(const float* const* src, const int64_t* ld, const int64_t* const* idx, const int64_t* stride,
                      const int64_t* rows, int32_t n_pieces, int64_t n_out, int32_t D, float* out, int64_t ldo,
                      int32_t* err_flag, spk_stream_t stream);
int spk_mlp_head_fwd(const float* H1, int64_t ldh, const float* b1, const float* w2, const float* b2, float slope,
                     int64_t n_rows, int32_t D, float* out, spk_stream_t stream);
int spk_mlp_head_bwd(const float* H1, int64_t ldh, const float* b1, const float* w2, float slope, const float* dout,
                     int64_t n_rows, int32_t D, float* dH1, int64_t ldd, float* act, int64_t lda, spk_stream_t stream);
int spk_tanh_fwd(float* x, int64_t ld, int64_t n_rows, int32_t width, spk_stream_t stream);
int spk_tanh_bwd(const float* y, int64_t ldy, const float* dout, int64_t ldo, int64_t n_rows, int32_t width, float* dpre,
                 int64_t ldp, spk_stream_t stream);
int spk_rank_scores(const float* U, int64_t ldu, const float* Bt, int64_t ldb, const float* w2, const float* b2, float slope,
                    int64_t n_pairs, int32_t n_rel, int32_t D, float* out, int64_t ldo, spk_stream_t stream);

/* ---- ConvKB link-prediction evaluation: filtered entity ranks (Corpus.get_validation_pred, GAT/create_batch.py:905-1199) --
 * AC [N, 2D] (row stride ldac >= 2D) = [A | C] = E . [W1a^T | W1c^T], Bt [R, D] = Rel . W1b^T, b1 / w2 = fc1.bias / fc2.weight
 * (fc2.bias is dropped: it shifts every score of a row alike). side 0 ranks heads: candidates (c, r, t), pair vector
 * v_i = C[t_i] + Bt[r_i] + b1, candidate rows A[c]; side 1 ranks tails: (h, r, c), v_i = A[h_i] + Bt[r_i] + b1, rows C[c].
 * s_c = sum_{d=0..D-1} w2[d] * lrelu(X[c,d] + v_i[d]) as one sequential fp32 chain in every kernel (so a score is the same
 * float wherever it is computed); 1 <= D <= 512, 0 <= slope <= 1. a > b below means a > b or (isnan(a) && !isnan(b)).
 * spk_linkpred_count:  for the test triples int64 [T,3] (h, r, t) writes V [T, ldv >= D] = v_i, true_id int32 [T] = the
 *                      ranked entity (-1 when keep[i] == 0 or an id is out of range; keep uint8 [T] may be null = keep all),
 *                      s_true float [T] and count int32 [T] = #{c in [0,N), c != true_id[i] : s_c > s_true[i]}; the
 *                      T x N scores are never stored. An id outside [0, N) / [0, R) sets bit 0 of *err_flag.
 * spk_linkpred_filter: after spk_linkpred_count on the same arguments and stream: keys int64 [n_keys] are the sorted,
 *                      possibly repeated spk_triple_keys of the known triples, in (h, r, t) order for side 1 and of the
 *                      column-swapped (t, r, h) triples for side 0, so row i's known candidates are one key range;
 *                      subtracts from count[i] each distinct known candidate c != true_id[i] with s_c > s_true[i].
 *                      work: int64 [3T + 1] scratch. A decoded id outside [0, N) sets bit 1 of *err_flag.
 * The filtered rank of row i is 1 + count[i] (the position of the test triple under a stable descending sort). */
int spk_linkpred_count(const float* AC, int64_t ldac, int64_t n_ent, const float* Bt, int64_t ldb, int64_t n_rel,
                       const float* b1, const float* w2, float slope, int32_t D, const int64_t* triples,
                       const uint8_t* keep, int64_t n_pairs, int32_t side, float* V, int64_t ldv, float* s_true,
                       int32_t* true_id, int32_t* count, int32_t* err_flag, spk_stream_t stream);
int spk_linkpred_filter(const float* AC, int64_t ldac, int64_t n_ent, int64_t n_rel, const float* w2, float slope,
                        int32_t D, const int64_t* triples, int64_t n_pairs, int32_t side, const float* V, int64_t ldv,
                        const float* s_true, const int32_t* true_id, const int64_t* keys, int64_t n_keys, int64_t* work,
                        int32_t* count, int32_t* err_flag, spk_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* SPKBGAT_H */
