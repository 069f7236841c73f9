"""autograd.Function shells around the libspkbgat kernels.

Math (SURVEY.md 8 a-4 / a-5), per attention-layer group with heads h, a_h = [A1|A2|A3], a_2,h:
    P1 = X A1^T, P2 = X A2^T, P3 = Rel A3^T,  q* = P* a_2^T      (projection GEMMs, K1)
    m_e = P1[i] + P2[j] + P3[k](+P3[k2]),  s_e = q1[i] + q2[j] + q3[k](+q3[k2])
    ee_e = exp(-LeakyReLU(s_e)),  out_i = ELU( sum_e msk_e ee_e m_e / sum_e ee_e )   (K2)
which is GAT/layers.py:124-175 with the a.mm(edge_h) product re-associated so that no E-sized
feature tensor exists. The weights are handed to the kernels as "extended" matrices
    Wn [F, 2*Wd] = [A1^T | A1^T a_2^T | 0 || A2^T | A2^T a_2^T | 0],   Wr [Rd, Wd] = [A3^T | A3^T a_2^T | 0]
built from the reference-shaped parameters `a`, `a_2` with differentiable torch ops on these tiny
tensors, so autograd chains dWn, dWr back to a and a_2.
"""
import ctypes as C
import os
import weakref

import torch

from . import _lib
from .graph import KGraph

MAX_HEADS = 4
USE_TC = True          # route eligible products through the tcgen05 3xTF32 GEMM (else the exact-fp32 SIMT GEMM)
TC_MIN_ROWS = 1        # (tests lower/raise this to exercise both paths)


WD_ALIGN = int(os.environ.get("SPK_WD_ALIGN", "8"))     # projected-row width granularity in floats (8 = one 32-byte sector)


class Geometry:
    """Row format of the projected tables for H heads of width D (see include/spkbgat.h)."""

    def __init__(self, n_heads, d_head):
        assert 1 <= n_heads <= MAX_HEADS
        self.H, self.D = n_heads, d_head
        self.Dp = (d_head + 3) // 4 * 4
        self.Dt = self.H * self.Dp
        self.Wd = (self.Dt + self.H + WD_ALIGN - 1) // WD_ALIGN * WD_ALIGN
        if self.Wd > 512 and WD_ALIGN > 8:
            self.Wd = (self.Dt + self.H + 7) // 8 * 8
        if self.Wd > 512:
            raise ValueError(f"heads*out_features = {n_heads}*{d_head} exceeds the 512-float fused row")

    def struct(self):
        return _lib.Geom(self.H, self.D, self.Dp, self.Wd)


class AttnWeightsFn(torch.autograd.Function):
    """(a_0 .. a_{H-1}, a_2,0 .. a_2,{H-1}) -> the extended weight matrices of one head group, on the library's assembly
    kernels (spk_attn_weights_fwd / _bwd): mode 0 -> (Wn, Wr), mode 1 -> (Wa, V, V3). Same values and gradients as the
    torch formulation below (`_extended_weights_torch`, `_agg_weights_torch`: kept for CPU tensors / fp64 checks)."""

    @staticmethod
    def _args(mode, dims, params):
        H = len(params) // 2
        w = _lib.AttnWeightsArgs()
        for h in range(H):
            w.a[h] = params[h].data_ptr(); w.a2[h] = params[H + h].data_ptr()
        w.n_heads = H; w.F, w.Rd, w.D = dims["F"], dims["Rd"], dims["D"]
        w.mode = mode
        if mode == 0:
            w.d_pad, w.width = dims["Dp"], dims["Wd"]
        else:
            w.f_pad, w.lz = dims["Fp"], dims["LZ"]
        return w

    @staticmethod
    def forward(ctx, mode, dims, *params):
        params = tuple(p.contiguous() for p in params)
        dev = params[0].device
        f32 = dict(dtype=torch.float32, device=dev)
        F, Rd, D, H = dims["F"], dims["Rd"], dims["D"], len(params) // 2
        if mode == 0:
            outs = (torch.empty(F, 2 * dims["Wd"], **f32), torch.empty(Rd, dims["Wd"], **f32))
        else:
            outs = (torch.empty(H, dims["LZ"], D, **f32), torch.empty(F, 4, **f32), torch.empty(Rd, 4, **f32))
        w = AttnWeightsFn._args(mode, dims, params)
        w.W0 = outs[0].data_ptr(); w.ld0 = outs[0].stride(0) if mode == 0 else D
        w.W1 = outs[1].data_ptr(); w.ld1 = outs[1].stride(0)
        if mode == 1:
            w.W2 = outs[2].data_ptr()
        _lib.check(_lib.load().spk_attn_weights_fwd(C.byref(w), _lib.stream_ptr()), "attn_weights_fwd")
        ctx.save_for_backward(*params)
        ctx.mode, ctx.dims = mode, dims
        return outs

    @staticmethod
    def backward(ctx, *grads):
        params = ctx.saved_tensors
        mode, dims = ctx.mode, ctx.dims
        dev = params[0].device
        F, Rd, D, H = dims["F"], dims["Rd"], dims["D"], len(params) // 2
        shapes = ((F, 2 * dims["Wd"]), (Rd, dims["Wd"])) if mode == 0 else ((H, dims["LZ"], D), (F, 4), (Rd, 4))
        g = [torch.zeros(s, dtype=torch.float32, device=dev) if x is None else x.contiguous() for x, s in zip(grads, shapes)]
        dparams = [torch.empty_like(p) for p in params]
        w = AttnWeightsFn._args(mode, dims, params)
        for h in range(H):
            w.da[h] = dparams[h].data_ptr(); w.da2[h] = dparams[H + h].data_ptr()
        w.W0 = g[0].data_ptr(); w.ld0 = g[0].stride(0) if mode == 0 else D
        w.W1 = g[1].data_ptr(); w.ld1 = g[1].stride(0)
        if mode == 1:
            w.W2 = g[2].data_ptr()
        _lib.check(_lib.load().spk_attn_weights_bwd(C.byref(w), _lib.stream_ptr()), "attn_weights_bwd")
        return (None, None) + tuple(dparams)


def _on_library(tensors):
    return all(t.is_cuda and t.dtype == torch.float32 for t in tensors)


def extended_weights(a_list, a2_list, in_features, geom):
    """a_list[h]: [D, 2F+Rd], a2_list[h]: [1, D] (GAT/layers.py:100-105) -> Wn [F, 2Wd], Wr [Rd, Wd]."""
    if _on_library(list(a_list) + list(a2_list)):
        dims = dict(F=in_features, Rd=a_list[0].shape[1] - 2 * in_features, D=geom.D, Dp=geom.Dp, Wd=geom.Wd)
        return AttnWeightsFn.apply(0, dims, *a_list, *a2_list)
    return _extended_weights_torch(a_list, a2_list, in_features, geom)


def _extended_weights_torch(a_list, a2_list, in_features, geom):
    F = in_features
    a0 = a_list[0]
    rd = a0.shape[1] - 2 * F
    Wn = a0.new_zeros(F, 2 * geom.Wd)
    Wr = a0.new_zeros(rd, geom.Wd)
    for h, (a, a2) in enumerate(zip(a_list, a2_list)):
        lo = h * geom.Dp
        at = a.t()                                       # [2F+Rd, D]
        qa = (at * a2).sum(dim=1)                        # [2F+Rd]  = a^T a_2^T (elementwise: no library GEMV on the path)
        Wn[:, lo:lo + geom.D] = at[:F]
        Wn[:, geom.Dt + h] = qa[:F]
        Wn[:, geom.Wd + lo:geom.Wd + lo + geom.D] = at[F:2 * F]
        Wn[:, geom.Wd + geom.Dt + h] = qa[F:2 * F]
        Wr[:, lo:lo + geom.D] = at[2 * F:]
        Wr[:, geom.Dt + h] = qa[2 * F:]
    return Wn, Wr


# ---- dense products --------------------------------------------------------------------------

def gemm_nn(A, B, out=None, accumulate=False, act=0):
    """out[M,N] (+)= A[M,K] @ B[K,N] on the library's GEMM (row-major, last-dim contiguous views allowed).
    act=1 applies ELU, act=2 tanh to the final value (fused into the tensor-core epilogue)."""
    assert A.dim() == 2 and B.dim() == 2 and A.shape[1] == B.shape[0]
    assert A.stride(1) == 1 and B.stride(1) == 1
    M, K = A.shape
    N = B.shape[1]
    if out is None:
        assert not accumulate
        # row stride padded to 16 B so the epilogue can store whole 128 B row segments by TMA
        out = torch.empty(M, (N + 3) // 4 * 4, dtype=torch.float32, device=A.device)[:, :N]
    assert out.stride(1) == 1 and out.shape[0] == M and out.shape[1] == N
    if M and N:
        lib = _lib.load()
        if lib.timing is not None:
            _lib.current_tag = f"{M}x{K}x{N}"
        if K == 0:
            if not accumulate:
                out.zero_()
        elif USE_TC and M >= TC_MIN_ROWS and N <= 512 and lib.spk_gemm_nn_tc_supported(_lib.ptr(A), A.stride(0), M, N, K):
            # tcgen05 tensor cores, 3xTF32 (fp32-accurate)
            ws = torch.empty(lib.spk_gemm_tc_workspace_floats(N, K), dtype=torch.float32, device=A.device)
            _lib.check(lib.spk_gemm_nn_tc_act(_lib.ptr(A), A.stride(0), _lib.ptr(B), B.stride(0), _lib.ptr(out),
                                              out.stride(0), M, N, K, int(accumulate), int(act), _lib.ptr(ws),
                                              _lib.stream_ptr()), "gemm_nn_tc")
            return out
        else:
            _lib.check(lib.spk_gemm_nn(_lib.ptr(A), A.stride(0), _lib.ptr(B), B.stride(0), _lib.ptr(out),
                                       out.stride(0), M, N, K, int(accumulate), _lib.stream_ptr()), "gemm_nn")
        if act == 2:
            _lib.check(lib.spk_tanh_fwd(_lib.ptr(out), out.stride(0), M, N, _lib.stream_ptr()), "tanh_fwd")
        elif act:
            _lib.check(lib.spk_elu_inplace(_lib.ptr(out), out.stride(0), M, N, _lib.stream_ptr()), "elu_inplace")
    return out


def gemm_tn(A, B, out=None, accumulate=False):
    """out[Ka,Nb] (+)= A[M,Ka]^T @ B[M,Nb], deterministic fixed-order split over M."""
    assert A.dim() == 2 and B.dim() == 2 and A.shape[0] == B.shape[0]
    assert A.stride(1) == 1 and B.stride(1) == 1
    M, Ka = A.shape
    Nb = B.shape[1]
    lib = _lib.load()
    if out is None:
        assert not accumulate
        out = torch.empty(Ka, Nb, dtype=torch.float32, device=A.device)
    if Ka and Nb:
        if lib.timing is not None:
            _lib.current_tag = f"{M}x{Ka}x{Nb}"
        if USE_TC and M >= TC_MIN_ROWS and lib.spk_gemm_tn_tc_supported(_lib.ptr(A), A.stride(0), _lib.ptr(B), B.stride(0),
                                                                        M, Ka, Nb):
            ws = torch.empty(max(1, lib.spk_gemm_tn_tc_workspace_floats(M, Ka, Nb)), dtype=torch.float32, device=A.device)
            _lib.check(lib.spk_gemm_tn_tc(_lib.ptr(A), A.stride(0), _lib.ptr(B), B.stride(0), _lib.ptr(out),
                                          out.stride(0), M, Ka, Nb, int(accumulate), _lib.ptr(ws), _lib.stream_ptr()),
                       "gemm_tn_tc")
        else:
            ws = torch.empty(max(1, lib.spk_gemm_tn_workspace_floats(M, Ka, Nb)), dtype=torch.float32, device=A.device)
            _lib.check(lib.spk_gemm_tn(_lib.ptr(A), A.stride(0), _lib.ptr(B), B.stride(0), _lib.ptr(out), out.stride(0),
                                       M, Ka, Nb, int(accumulate), _lib.ptr(ws), _lib.stream_ptr()), "gemm_tn")
    return out


def tc_friendly(X):
    """Row stride multiple of 4 floats (16 B) so TMA can fetch the operand; pads a copy when needed."""
    if X.dim() != 2 or X.stride(1) != 1 or X.stride(0) % 4 == 0 or not USE_TC:
        return X
    f = X.shape[1]
    Xp = X.new_zeros(X.shape[0], (f + 3) // 4 * 4)
    Xp[:, :f] = X
    return Xp[:, :f]


# The aggregate-then-project layer builds a table whose rows START with the input row x at a 16-byte aligned stride
# (X~ = [x | pad | score scalars]); a later X @ W on the same tensor (entity_embeddings.mm(W_entities), models.py:175) reads
# its operand from that table instead of making a padded copy of the [N, 50] matrix for TMA (0.33 ms per step at C2).
_X_TABLE = {"key": None, "table": None}


def _x_key(X):
    return (X.data_ptr(), X._version, tuple(X.shape), tuple(X.stride()), str(X.device))


def _tma_operand(X):
    if _X_TABLE["key"] is not None and _X_TABLE["key"] == _x_key(X) and USE_TC:
        t = _X_TABLE["table"]()                             # weak reference: the cache never keeps the table alive
        _X_TABLE["key"] = _X_TABLE["table"] = None          # one-shot: the table is only trusted right after it was built
        if t is not None:
            return t[:, :X.shape[1]]
    return tc_friendly(X.contiguous())


class MatMulFn(torch.autograd.Function):
    """X @ W with the library GEMMs (relation_embed.mm(W) models.py:77, entity_embeddings.mm(W_entities) 175)."""

    @staticmethod
    def forward(ctx, X, W, dist=None):
        X = _tma_operand(X); W = W.contiguous()
        ctx.save_for_backward(X, W)
        ctx.dist = dist
        return gemm_nn(X, W)

    @staticmethod
    def backward(ctx, g):
        X, W = ctx.saved_tensors
        g = g.contiguous()
        dX = gemm_nn(g, W.t().contiguous()) if ctx.needs_input_grad[0] else None
        dW = gemm_tn(X, g) if ctx.needs_input_grad[1] else None
        if dW is not None and ctx.dist is not None:
            ctx.dist.all_reduce(dW)          # X rows are partitioned across ranks
        return dX, dW, None


def matmul(X, W, dist=None):
    """dist: DistContext when X's rows are partitioned across ranks (dW is then all-reduced)."""
    return MatMulFn.apply(X, W, dist)


# ---- fused attention-layer group -------------------------------------------------------------

def _hub_partial(hubs, ldpart, device):
    if hubs is None or hubs.n_tasks == 0:
        return None
    return torch.empty(hubs.n_tasks, ldpart, dtype=torch.float32, device=device)


def edge_attn_forward(graph, P1, P2, P3, geom, alpha, apply_elu, mask_csr, nanflag, elu_rows=0):
    """K2 launch. P1/P2: [n, >=Wd] views with unit inner stride; returns (out [N,H*D], den [N,H], sw [N,H]).
    elu_rows > 0: the ELU is applied to rows < elu_rows only."""
    lib = _lib.load()
    n = graph.n_nodes
    dev = P1.device
    out = torch.empty(n, geom.H * geom.D, dtype=torch.float32, device=dev)
    den = torch.empty(n, geom.H, dtype=torch.float32, device=dev)
    sw = torch.empty(n, geom.H, dtype=torch.float32, device=dev)
    a = _lib.EdgeFwdArgs()
    a.segptr = graph.rowptr.data_ptr(); a.col = graph.col.data_ptr(); a.t1 = graph.t1.data_ptr()
    a.t2 = graph.t2.data_ptr() if graph.t2 is not None else None
    a.P1 = P1.data_ptr(); a.ld1 = P1.stride(0)
    a.P2 = P2.data_ptr(); a.ld2 = P2.stride(0)
    a.P3 = P3.data_ptr(); a.ld3 = P3.stride(0)
    if mask_csr is not None:
        a.mask = mask_csr.data_ptr(); a.mask_stride = mask_csr.stride(0)
    a.out = out.data_ptr(); a.ldo = out.stride(0); a.den = den.data_ptr(); a.sw = sw.data_ptr()
    a.nanflag = nanflag.data_ptr()
    a.n_rows = n; a.apply_elu = int(apply_elu); a.alpha = float(alpha); a.elu_rows = int(elu_rows)
    a.geom = geom.struct()
    ldpart = geom.Wd + 2 * MAX_HEADS
    partial = _hub_partial(graph.row_hubs, ldpart, dev)
    graph.row_hubs.fill(a.hub, partial, ldpart)
    _lib.check(lib.spk_edge_attn_fwd(C.byref(a), _lib.stream_ptr()), "edge_attn_fwd")
    return out, den, sw


# Backward schedule of the projected layer groups:
#   "split": node pass + column pass + relation pass with the per-edge dot split between them (K3"/K4", no 2-hop edges)
#   "fused": node pass + one column pass that also gathers P3~[k] (K3'/K4'), relation pass = K4
#   "rows" : K3 over the rows, then K4 over columns and relations
# "split" falls back to "rows" for graphs with 2-hop edges.
BWD_MODE = os.environ.get("SPK_BWD_MODE", "split")


def _fill_fused_args(f, graph, P1, P2, P3, geom, alpha, apply_elu, mask_csr, out, dout, den, sw, G, ldg, rowsc, dP1, dP2, rec):
    f.rowptr = graph.rowptr.data_ptr()
    f.colptr = graph.colptr.data_ptr(); f.csc_row = graph.csc_row.data_ptr(); f.csc_pos = graph.csc_pos.data_ptr()
    f.csc_t1 = graph.csc_t1.data_ptr(); f.csc_t2 = graph.csc_t2.data_ptr() if graph.csc_t2 is not None else None
    f.P1 = P1.data_ptr(); f.ld1 = P1.stride(0); f.P2 = P2.data_ptr(); f.ld2 = P2.stride(0)
    f.P3 = P3.data_ptr(); f.ld3 = P3.stride(0)
    if mask_csr is not None:
        f.mask = mask_csr.data_ptr(); f.mask_stride = mask_csr.stride(0)
    f.out = out.data_ptr(); f.dout = dout.data_ptr(); f.ldo = out.stride(0)
    assert dout.stride(0) == out.stride(0)
    f.den = den.data_ptr(); f.sw = sw.data_ptr()
    f.G = G.data_ptr(); f.ldg = ldg; f.rowsc = rowsc.data_ptr()
    f.dP1 = dP1.data_ptr(); f.ldd1 = dP1.stride(0); f.dP2 = dP2.data_ptr(); f.ldd2 = dP2.stride(0)
    f.rec = rec.data_ptr() if rec is not None else None
    f.n_rows = graph.n_nodes; f.n_cols = graph.n_cols; f.apply_elu = int(apply_elu); f.alpha = float(alpha)
    f.geom = geom.struct()
    graph.row_hubs.fill(f.row_hub, None, 0)
    part = _hub_partial(graph.col_hubs, geom.Wd, P1.device)
    graph.col_hubs.fill(f.col_hub, part, geom.Wd)
    return part


def edge_attn_backward(graph, P1, P2, P3, geom, alpha, apply_elu, mask_csr, out, dout, den, sw, dP1, dP2, dP3,
                       after_columns=None, colsum=None):
    """Backward edge passes. Fills dP1 [n_rows, Wd], dP2 [n_cols, Wd] (indexed by gathered node) and dP3 [R, Wd].
    Multi-GPU hook: `after_columns()` is called as soon as dP2 is complete except for its q slot (the column sums of ds,
    which need the relation pass); those sums then go to `colsum` [n_cols, H]. Returns True when that split happened,
    False when dP2 came out complete in one piece (schedules other than "split")."""
    lib = _lib.load()
    graph.build_backward()
    n, dev = graph.n_nodes, P1.device
    ldg = _row_stride(geom.Dt, G_ALIGN)
    G = torch.empty(n, ldg, dtype=torch.float32, device=dev)
    mode = BWD_MODE if sw is not None else "rows"
    if mode == "split" and graph.t2 is not None:
        mode = "rows"
    ne = max(1, graph.n_edges)
    if mode == "split":
        q = _lib.EdgeBwdSplitArgs()
        rowsc = torch.empty(max(1, n), geom.H, 4, dtype=torch.float32, device=dev)
        rec4 = torch.empty(ne, geom.H, 4, dtype=torch.float32, device=dev)
        dsv = torch.empty(ne, geom.H, dtype=torch.float32, device=dev)
        keep = _fill_fused_args(q.base, graph, P1, P2, P3, geom, alpha, apply_elu, mask_csr, out, dout, den, sw, G, ldg,
                                rowsc, dP1, dP2, None)
        q.relptr = graph.relptr.data_ptr(); q.rel_row = graph.rel_row.data_ptr(); q.rel_pos = graph.rel_pos.data_ptr()
        q.rec4 = rec4.data_ptr(); q.dsv = dsv.data_ptr()
        q.dP3 = dP3.data_ptr(); q.ldd3 = dP3.stride(0); q.n_rel = graph.n_rel
        part3 = _hub_partial(graph.rel_hubs, geom.Wd, dev)
        graph.rel_hubs.fill(q.rel_hub, part3, geom.Wd)
        part1 = _hub_partial(graph.row_hubs, 4, dev)                # row sums of ds over hub rows
        graph.row_hubs.fill(q.base.row_hub, part1, 4)
        if after_columns is None:
            if lib.timing is None:
                _lib.check(lib.spk_edge_attn_bwd_split(C.byref(q), _lib.stream_ptr()), "edge_attn_bwd_split")
            else:                           # bench.py's per-kernel timing pass: one pass (= one gather kernel) per call
                for ph, tag in ((1, "node"), (2, "cols"), (4, "rels"), (8, "colsums")):
                    q.phases = ph
                    _lib.current_tag = tag
                    _lib.check(lib.spk_edge_attn_bwd_split(C.byref(q), _lib.stream_ptr()), "edge_attn_bwd_split")
                _lib.current_tag = ""
            del keep, part3, part1
            return False
        q.phases = 3
        _lib.current_tag = "node+cols"
        _lib.check(lib.spk_edge_attn_bwd_split(C.byref(q), _lib.stream_ptr()), "edge_attn_bwd_split")
        after_columns()
        q.phases = 12
        q.colsum = colsum.data_ptr(); q.ld_colsum = colsum.stride(0)
        _lib.current_tag = "rels+sums"
        _lib.check(lib.spk_edge_attn_bwd_split(C.byref(q), _lib.stream_ptr()), "edge_attn_bwd_split")
        _lib.current_tag = ""
        del keep, part3, part1
        return True
    rec = torch.empty(ne, 2 * geom.H, dtype=torch.float32, device=dev)
    if mode == "fused":
        f = _lib.EdgeBwdFusedArgs()
        rowsc = torch.empty(max(1, n), geom.H, 4, dtype=torch.float32, device=dev)
        keep = _fill_fused_args(f, graph, P1, P2, P3, geom, alpha, apply_elu, mask_csr, out, dout, den, sw, G, ldg, rowsc,
                                dP1, dP2, rec)
        _lib.check(lib.spk_edge_attn_bwd_fused(C.byref(f), _lib.stream_ptr()), "edge_attn_bwd_fused")
        del keep
        seg_gather(graph.relptr, graph.rel_row, graph.rel_pos, graph.rel_hubs, G, ldg, rec, geom, dP3, graph.n_rel, "rels")
        return False
    a = _lib.EdgeBwdRowsArgs()
    a.segptr = graph.rowptr.data_ptr(); a.col = graph.col.data_ptr(); a.t1 = graph.t1.data_ptr()
    a.t2 = graph.t2.data_ptr() if graph.t2 is not None else None
    a.P1 = P1.data_ptr(); a.ld1 = P1.stride(0)
    a.P2 = P2.data_ptr(); a.ld2 = P2.stride(0)
    a.P3 = P3.data_ptr(); a.ld3 = P3.stride(0)
    if mask_csr is not None:
        a.mask = mask_csr.data_ptr(); a.mask_stride = mask_csr.stride(0)
    a.out = out.data_ptr(); a.dout = dout.data_ptr(); a.ldo = out.stride(0)
    assert dout.stride(0) == out.stride(0)
    a.den = den.data_ptr()
    a.G = G.data_ptr(); a.ldg = ldg; a.dP1 = dP1.data_ptr(); a.ldd1 = dP1.stride(0); a.rec = rec.data_ptr()
    a.n_rows = n; a.apply_elu = int(apply_elu); a.alpha = float(alpha)
    a.geom = geom.struct()
    part_a = _hub_partial(graph.row_hubs, 2 * MAX_HEADS, dev)
    graph.row_hubs.fill(a.hub, part_a, 2 * MAX_HEADS)
    _lib.check(lib.spk_edge_attn_bwd_rows(C.byref(a), _lib.stream_ptr()), "edge_attn_bwd_rows")

    seg_gather(graph.colptr, graph.csc_row, graph.csc_pos, graph.col_hubs, G, ldg, rec, geom, dP2, graph.n_cols, "cols")
    seg_gather(graph.relptr, graph.rel_row, graph.rel_pos, graph.rel_hubs, G, ldg, rec, geom, dP3, graph.n_rel, "rels")
    return False


def seg_gather(ptr, src, pos, hubs, G, ldg, rec, geom, dst, n_seg, tag):
    """K4 launch: dst[seg] = [ sum_e w_e,h G[src_e] (per head chunk) | sum_e ds_e,h | 0 ] over the segments of `ptr`."""
    s = _lib.SegGatherArgs()
    s.segptr = ptr.data_ptr(); s.src = src.data_ptr(); s.pos = pos.data_ptr()
    s.G = G.data_ptr(); s.ldg = ldg; s.rec = rec.data_ptr()
    s.out = dst.data_ptr(); s.ldout = dst.stride(0); s.n_seg = n_seg
    s.flags = 1 if (n_seg > 0 and src.numel() < 5 * n_seg) else 0        # many short segments -> streaming kernel
    s.geom = geom.struct()
    part = _hub_partial(hubs, geom.Wd, G.device)
    hubs.fill(s.hub, part, geom.Wd)
    _lib.current_tag = f"{tag}:w{geom.Wd}"
    try:
        _lib.check(_lib.load().spk_edge_attn_bwd_segments(C.byref(s), _lib.stream_ptr()), "edge_attn_bwd_segments")
    finally:
        _lib.current_tag = ""


def _ghost_combine(ghost, vals, den, sw, n, H):
    """Hub rows split across ranks (dist.RowPartition): rows n.. of `vals` [n_ext, H*W] hold this rank's slice result
    normalised by its own denominator (num_loc / den_loc), `den` / `sw` [n_ext, H] the slice sums. Recovers the
    un-normalised partials, sums them over the ranks (GAT/layers.py:150-169 is linear in the edges up to the final
    division) and writes num / den and den back; sw keeps the LOCAL slice sum (the backward wants the partial)."""
    ng = ghost.n
    W = vals.shape[1] // H
    v = vals[n:].view(ng, H, W)
    d = den[n:]
    d0 = torch.where(sw[n:] == 0, torch.zeros_like(d), d)           # an empty slice reports den = 1e-12 (layers.py:152)
    buf = torch.cat(((v * d0.unsqueeze(-1)).reshape(ng, H * W), d0), dim=1)
    ghost.sum_partials(buf)
    dg = buf[:, H * W:]
    dg = torch.where(dg == 0, torch.full_like(dg, 1e-12), dg)
    vals[n:] = (buf[:, :H * W].view(ng, H, W) / dg.unsqueeze(-1)).reshape(ng, H * W)
    den[n:] = dg


def _ghost_dout(ghost, dout, n, n_ext):
    """[n, W] gradient of this rank's rows -> [n_ext, W]: ghost rows get the owners' gradient rows (on every rank), the
    owner's own (edge-less) copy of a hub row gets zero: its gradient flows through the ghost row."""
    ext = torch.empty(n_ext, dout.shape[1], dtype=dout.dtype, device=dout.device)
    ext[:n] = dout
    ext[n:] = ghost.gather_rows(dout)
    ext[ghost.mine_local] = 0
    return ext


class AttentionGroupFn(torch.autograd.Function):
    """One fused group of <=4 heads: (X, Wn, Rel, Wr) -> ELU?(attention output) [N, H*D].

    Multi-GPU (graph.dist set, SURVEY.md 8e): rows are partitioned; the gathered table P2~ must cover all nodes.
      * "proj"  exchange: all-gather the projected rows P2~ [n, Wd]; backward reduce-scatters the partial dP2~.
      * "input" exchange (chosen when the input is narrower than the projection, i.e. layer 1: F=50 vs Wd=208):
        all-gather X [n, F] and project all nodes locally (cheap on the tensor cores); backward projects the partial
        dP2~ back to input space and reduce-scatters [n, F]. 4x fewer bytes over NVLink for layer 1.
    """

    @staticmethod
    def forward(ctx, X, Wn, Rel, Wr, graph, geom, alpha, apply_elu, mask_csr, nanflag):
        X = tc_friendly(X.contiguous()); Wn = Wn.contiguous(); Rel = Rel.contiguous(); Wr = Wr.contiguous()
        dist = getattr(graph, "dist", None)
        ghost = dist.ghost if dist is not None else None
        Wd = geom.Wd
        mode = "local"
        X_all = None
        if dist is None:
            P3 = gemm_nn(Rel, Wr)               # [R, Wd]
            P = gemm_nn(X, Wn)                  # [N, 2Wd] = [P1~ | P2~]
            P1, P2 = P[:, :Wd], P[:, Wd:]
        elif 2 * X.shape[1] <= Wd:
            mode = "input"                      # every rank projects all nodes from the gathered input rows
            Fp = (X.shape[1] + 3) // 4 * 4
            X_all, mine = dist.gather_buffer(Fp, X.device)
            mine[:, :X.shape[1]].copy_(X)
            if Fp != X.shape[1]:
                mine[:, X.shape[1]:].zero_()
            h = dist.all_gather_start(X_all)
            P3 = gemm_nn(Rel, Wr)
            P1 = gemm_nn(X, Wn[:, :Wd])
            h.wait()
            X_all = X_all[:, :X.shape[1]]
            P2 = gemm_nn(X_all, Wn[:, Wd:])
        else:
            mode = "proj"                       # the GEMM writes this rank's P2~ rows straight into the exchange buffer
            P2, mine = dist.gather_buffer(Wd, X.device)
            gemm_nn(X, Wn[:, Wd:], out=mine)
            h = dist.all_gather_start(P2)       # in flight while P1~ and P3~ are projected
            n = X.shape[0]
            if ghost is None:
                P1 = gemm_nn(X, Wn[:, :Wd])
            else:                               # + the P1~ rows of the hub rows whose edges are split across ranks
                P1 = torch.empty(n + ghost.n, Wd, dtype=torch.float32, device=X.device)
                gemm_nn(X, Wn[:, :Wd], out=P1[:n])
                gemm_nn(tc_friendly(ghost.gather_rows(X)), Wn[:, :Wd], out=P1[n:])
            P3 = gemm_nn(Rel, Wr)
            h.wait()
        if ghost is not None and mode != "proj":
            raise NotImplementedError("hub rows split across ranks need the projected exchange (or the aggregate-then-project path)")
        if ghost is None:
            out, den, sw = edge_attn_forward(graph, P1, P2, P3, geom, alpha, apply_elu, mask_csr, nanflag)
            out_ret = out
        else:
            n = X.shape[0]
            # the kernel applies the ELU to this rank's own rows; the ghost rows behind them come out as num_loc / den_loc and
            # get theirs after the partial sums of all ranks are combined (a few rows, not a pass over the whole output)
            k_elu = bool(apply_elu) and n > 0                    # (a rank may own no rows at all: then every row is a ghost row)
            out, den, sw = edge_attn_forward(graph, P1, P2, P3, geom, alpha, k_elu, mask_csr, nanflag, elu_rows=n if k_elu else 0)
            _ghost_combine(ghost, out, den, sw, n, geom.H)
            nanflag.bitwise_or_(torch.isnan(out[n:]).any().to(torch.int32))
            if apply_elu and out.shape[0] > n:
                tail = out[n:]
                _lib.check(_lib.load().spk_elu_inplace(_lib.ptr(tail), tail.stride(0), tail.shape[0], tail.shape[1],
                                                       _lib.stream_ptr()), "elu_inplace")
            out[ghost.mine_local] = out[n:][ghost.mine]          # the owner's copy of a hub row takes the combined result
            out_ret = out[:n]
        ctx.save_for_backward(X, Wn, Rel, Wr, P1, P2, P3, out, den, sw, X_all if X_all is not None else X.new_empty(0))
        ctx.graph, ctx.geom, ctx.alpha, ctx.apply_elu, ctx.mask_csr, ctx.mode = graph, geom, alpha, apply_elu, mask_csr, mode
        ctx.mark_non_differentiable(den, sw)
        return out_ret, den, sw

    @staticmethod
    def backward(ctx, dout, _dden, _dsw):
        geom, graph, mode = ctx.geom, ctx.graph, ctx.mode
        dist = getattr(graph, "dist", None)
        X, Wn, Rel, Wr, P1, P2, P3, out, den, sw, X_all = ctx.saved_tensors
        Wd = geom.Wd
        dout = dout.contiguous()
        n = X.shape[0]
        dev = X.device
        dP3 = torch.empty_like(P3)
        WnT = Wn.t().contiguous()               # [2Wd, F]
        need_x, need_w = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        dX = dWn = None
        if mode == "local":
            dP = torch.empty(n, 2 * Wd, dtype=torch.float32, device=dev)
            edge_attn_backward(graph, P1, P2, P3, geom, ctx.alpha, ctx.apply_elu, ctx.mask_csr, out, dout, den, sw,
                               dP[:, :Wd], dP[:, Wd:], dP3)
            if need_x:
                dX = gemm_nn(dP, WnT)
            if need_w:
                dWn = gemm_tn(X, dP)
        else:
            # partial dP2~ over this rank's edges for ALL gathered nodes -> owners. "proj": reduce-scatter the projected
            # rows; "input": project the partial back to input space first (F < Wd floats per node over NVLink).
            # The reduce-scatter starts right after the column pass and runs under the relation pass and the products
            # that only need dP1~.
            mr = dist.part.max_rows
            ghost = dist.ghost
            n_ext = n + (ghost.n if ghost is not None else 0)
            if ghost is not None:
                dout = _ghost_dout(ghost, dout, n, n_ext)
            dP1 = torch.empty(n_ext, Wd, dtype=torch.float32, device=dev)
            dP2_all = torch.empty_like(P2)
            colsum = torch.empty(P2.shape[0], geom.H, dtype=torch.float32, device=dev)
            pend = {}

            def start_main():
                if mode == "proj":
                    pend["pad"] = torch.empty(mr, Wd, dtype=torch.float32, device=dev)
                    pend["h"] = dist.reduce_scatter_start(dP2_all, pend["pad"])

            split = edge_attn_backward(graph, P1, P2, P3, geom, ctx.alpha, ctx.apply_elu, ctx.mask_csr, out, dout, den, sw,
                                       dP1, dP2_all, dP3, after_columns=start_main if mode == "proj" else None, colsum=colsum)
            if mode == "proj":
                if split:
                    qs_pad = torch.empty(mr, geom.H, dtype=torch.float32, device=dev)
                    hq = dist.reduce_scatter_start(colsum, qs_pad)
                else:
                    start_main()
                h3 = dist.all_reduce_start(dP3)
                if ghost is not None:           # dP1~ of a hub row = sum of the ranks' partials -> its owner's row
                    gsum = ghost.sum_partials(dP1[n:].contiguous())
                    dP1[ghost.mine_local] = gsum[ghost.mine]
                    dP1 = dP1[:n]
                if need_x:
                    dX = gemm_nn(dP1, WnT[:Wd])
                if need_w:
                    dWn = torch.empty_like(Wn)
                    gemm_tn(X, dP1, out=dWn[:, :Wd])
                pend["h"].wait()
                dP2 = pend["pad"][:n]
                if split:
                    hq.wait()
                    dP2[:, geom.Dt:geom.Dt + geom.H].copy_(qs_pad[:n])
                del dP2_all
                if need_x:
                    gemm_nn(dP2, WnT[Wd:], out=dX, accumulate=True)
                if need_w:
                    gemm_tn(X, dP2, out=dWn[:, Wd:])
                    dist.all_reduce(dWn)
                h3.wait()
            else:                               # "input"
                h3 = dist.all_reduce_start(dP3)
                F = X.shape[1]
                Fp = (F + 3) // 4 * 4
                if need_x:
                    dX2_all = torch.empty(P2.shape[0], Fp, dtype=torch.float32, device=dev)
                    gemm_nn(dP2_all, WnT[Wd:], out=dX2_all[:, :F])
                    if Fp != F:
                        dX2_all[:, F:].zero_()
                    pad = torch.empty(mr, Fp, dtype=torch.float32, device=dev)
                    h = dist.reduce_scatter_start(dX2_all, pad)
                    dX1 = gemm_nn(dP1, WnT[:Wd])
                    h.wait()
                    dX = dX1.add_(pad[:n, :F])
                    del dX2_all
                if need_w:
                    dWn = torch.empty_like(Wn)
                    gemm_tn(X, dP1, out=dWn[:, :Wd])
                    gemm_tn(X_all, dP2_all, out=dWn[:, Wd:])
                    dist.all_reduce(dWn)
                h3.wait()
        dRel = gemm_nn(dP3, Wr.t().contiguous()) if ctx.needs_input_grad[2] else None
        dWr = gemm_tn(Rel, dP3) if ctx.needs_input_grad[3] else None
        return dX, dWn, dRel, dWr, None, None, None, None, None, None


# ---- aggregate-then-project variant (input narrower than the projection, i.e. layer 1) ---------

AGG_MODE = "auto"      # "auto": use it where it moves fewer bytes; "off": never; "force": wherever the shape is supported
AGG_BWD_MODE = os.environ.get("SPK_AGG_BWD_MODE", "split")     # "split": split-dot column / relation passes; "rows": round-1 schedule
AGG_MAX_HEADS = 2


# Row strides (floats) of the tables that are gathered one row per edge; the default keeps whole 32-byte sectors (8 floats),
# SPK_*_ALIGN = 16 / 32 rounds rows to 64 / 128 bytes so that a row never straddles one DRAM burst / cache line more than its
# size needs (more bytes per row, fewer partially used lines).
G_ALIGN = int(os.environ.get("SPK_G_ALIGN", "8"))
GX_ALIGN = int(os.environ.get("SPK_GX_ALIGN", "8"))
LX_ALIGN = int(os.environ.get("SPK_LX_ALIGN", "8"))


def _row_stride(width, align):
    return (width + align - 1) // align * align


class AggGeometry:
    """Shapes of the aggregate-then-project path (csrc/spk_agg.cuh): table rows [x | pad | 4 scalars | pad]."""

    def __init__(self, n_heads, in_features, nrela_dim, d_head):
        self.H, self.F, self.Rd, self.D = n_heads, in_features, nrela_dim, d_head
        self.Fx4, self.Fr4 = (in_features + 3) // 4, (nrela_dim + 3) // 4
        self.Fp, self.Rp = 4 * self.Fx4, 4 * self.Fr4
        self.LX = _row_stride(self.Fp + 4, LX_ALIGN)
        self.LR = _row_stride(self.Rp + 4, LX_ALIGN)
        self.LZ = 2 * self.Fp + self.Rp

    @staticmethod
    def supported(n_heads, in_features, nrela_dim):
        return 1 <= n_heads <= AGG_MAX_HEADS and 1 <= in_features <= 60 and 1 <= nrela_dim <= 60

    def struct(self):
        return _lib.AggGeom(self.H, self.Fx4, self.Fr4, self.LZ)


def use_agg_path(n_heads, in_features, nrela_dim, d_head, graph):
    if AGG_MODE == "off" or (getattr(graph, "dist", None) is None and graph.n_cols != graph.n_nodes):
        return False
    if not AggGeometry.supported(n_heads, in_features, nrela_dim):
        return False
    if AGG_MODE == "force":
        return True
    g = AggGeometry(n_heads, in_features, nrela_dim, d_head)
    return g.LX + g.LR < n_heads * d_head          # gathered bytes per edge: input rows vs one projected row


def agg_weights(a_list, a2_list, geom):
    """a_h [D, 2F+Rd], a_2,h [1, D] (GAT/layers.py:100-105) ->
         Wa [H, LZ, D]  a_h^T with zero rows at the pad positions of Zn_h = [sw x_i | sum w x_j | sum w r_k]
         V  [F, 4]      (A2^T a_2^T)_0, (..)_1, (A1^T a_2^T)_0, (..)_1      score vectors of X~
         V3 [Rd, 4]     (A3^T a_2^T)_0, (..)_1, 0, 0                        score vectors of Rel~
    On the library's assembly kernels for CUDA fp32 parameters (AttnWeightsFn), else differentiable torch ops."""
    if _on_library(list(a_list) + list(a2_list)):
        dims = dict(F=geom.F, Rd=geom.Rd, D=geom.D, Fp=geom.Fp, LZ=geom.LZ)
        return AttnWeightsFn.apply(1, dims, *a_list, *a2_list)
    return _agg_weights_torch(a_list, a2_list, geom)


def _agg_weights_torch(a_list, a2_list, geom):
    F, Rd, Fp = geom.F, geom.Rd, geom.Fp
    a0 = a_list[0]
    Wa = a0.new_zeros(geom.H, geom.LZ, geom.D)
    V = a0.new_zeros(F, 4)
    V3 = a0.new_zeros(Rd, 4)
    for h, (a, a2) in enumerate(zip(a_list, a2_list)):
        at = a.t()                                        # [2F+Rd, D]
        qa = (at * a2).sum(dim=1)                         # a^T a_2^T
        Wa[h, :F] = at[:F]
        Wa[h, Fp:Fp + F] = at[F:2 * F]
        Wa[h, 2 * Fp:2 * Fp + Rd] = at[2 * F:]
        V[:, 2 + h] = qa[:F]
        V[:, h] = qa[F:2 * F]
        V3[:, h] = qa[2 * F:]
    return Wa, V, V3


def _agg_table(X, V, ld, chunks, out=None):
    T = torch.empty(X.shape[0], ld, dtype=torch.float32, device=X.device) if out is None else out
    assert T.shape[0] == X.shape[0] and T.stride(1) == 1 and T.stride(0) >= ld
    ld = T.stride(0)
    if X.shape[0]:
        _lib.check(_lib.load().spk_agg_table(_lib.ptr(X), X.stride(0), _lib.ptr(V), _lib.ptr(T), ld, X.shape[0],
                                             X.shape[1], chunks, _lib.stream_ptr()), "agg_table")
    return T


class AggGroupFn(torch.autograd.Function):
    """One layer group on the aggregate-then-project kernels: (X, Rel, Wa, V, V3) -> ELU?(attention output) [N, H*D].
    Same math as AttentionGroupFn (GAT/layers.py:124-175), re-associated so the edges gather input rows."""

    @staticmethod
    def forward(ctx, X, Rel, Wa, V, V3, graph, geom, alpha, apply_elu, mask_csr, nanflag):
        lib = _lib.load()
        X = X.contiguous(); Rel = Rel.contiguous(); Wa = Wa.contiguous(); V = V.contiguous(); V3 = V3.contiguous()
        n, dev = graph.n_nodes, X.device
        n_loc = X.shape[0]
        H, D, LZ = geom.H, geom.D, geom.LZ
        dist = getattr(graph, "dist", None)
        ghost = dist.ghost if dist is not None else None
        # multi-GPU (SURVEY.md 8e): rows are partitioned, the gathered table must cover all nodes -> all-gather the
        # X~ rows (LX = 56 floats for F = 50: 3.7x fewer bytes than the projected rows). The table builder writes this
        # rank's rows straight into the exchange buffer; the all-gather runs in place, under the Rel~ table build.
        if dist is None:
            Xt = _agg_table(X, V, geom.LX, geom.Fx4)
            Xc = Xt
            Rt = _agg_table(Rel, V3, geom.LR, geom.Fr4)
            _X_TABLE["key"], _X_TABLE["table"] = _x_key(X), weakref.ref(Xt)
        else:
            Xc, Xt = dist.gather_buffer(geom.LX, dev)
            _agg_table(X, V, geom.LX, geom.Fx4, out=Xt)
            hx = dist.all_gather_start(Xc)
            Rt = _agg_table(Rel, V3, geom.LR, geom.Fr4)
            hx.wait()
            if ghost is not None:
                # hub rows split across ranks: their X~ rows arrived with the all-gather; park copies right after this
                # rank's own rows (spare rows of its slot: RowPartition.max_rows reserves them) so that the row table
                # [own rows | ghost rows] is one contiguous view of the exchange buffer
                lo = dist.rank * dist.part.max_rows
                Xc[lo + n_loc:lo + n] = Xc[ghost.padded_ids]
                Xt = Xc[lo:lo + n]
        Z = torch.empty(n, H * LZ, dtype=torch.float32, device=dev)
        den = torch.empty(n, H, dtype=torch.float32, device=dev)
        sw = torch.empty(n, H, dtype=torch.float32, device=dev)
        a = _lib.AggFwdArgs()
        a.segptr = graph.rowptr.data_ptr(); a.col = graph.col.data_ptr(); a.t1 = graph.t1.data_ptr()
        a.t2 = graph.t2.data_ptr() if graph.t2 is not None else None
        a.xrow = Xt.data_ptr(); a.ldxr = Xt.stride(0); a.xcol = Xc.data_ptr(); a.ldxc = Xc.stride(0)
        a.rel = Rt.data_ptr(); a.ldr = Rt.stride(0)
        if mask_csr is not None:
            a.mask = mask_csr.data_ptr(); a.mask_stride = mask_csr.stride(0)
        a.z = Z.data_ptr(); a.ldz = Z.stride(0); a.den = den.data_ptr(); a.sw = sw.data_ptr()
        a.nanflag = nanflag.data_ptr(); a.n_rows = n; a.alpha = float(alpha); a.geom = geom.struct()
        partial = _hub_partial(graph.row_hubs, 264, dev)
        graph.row_hubs.fill(a.hub, partial, 264)
        _lib.check(lib.spk_agg_fwd(C.byref(a), _lib.stream_ptr()), "agg_fwd")
        if ghost is not None:                               # Zn of a hub row: partial sums of every rank's edge slice
            _ghost_combine(ghost, Z, den, sw, n_loc, H)
        out = torch.empty(n, H * D, dtype=torch.float32, device=dev)
        for h in range(H):                                  # a.mm(.) of layers.py:137 on the aggregated rows (+ ELU 175)
            gemm_nn(Z[:, h * LZ:(h + 1) * LZ], Wa[h], out=out[:, h * D:(h + 1) * D], act=int(apply_elu))
        if ghost is not None:
            nanflag.bitwise_or_(torch.isnan(out[n_loc:]).any().to(torch.int32))
            out[ghost.mine_local] = out[n_loc:][ghost.mine]  # the owner's copy of a hub row takes the combined result
        ctx.save_for_backward(X, Rel, Wa, V, V3, Xt, Rt, Z, out, den, sw, Xc)
        ctx.graph, ctx.geom, ctx.alpha, ctx.apply_elu, ctx.mask_csr = graph, geom, alpha, apply_elu, mask_csr
        return out[:n_loc] if ghost is not None else out

    @staticmethod
    def backward(ctx, dout):
        lib = _lib.load()
        geom, graph = ctx.geom, ctx.graph
        X, Rel, Wa, V, V3, Xt, Rt, Z, out, den, sw, Xc = ctx.saved_tensors
        dist = getattr(graph, "dist", None)
        graph.build_backward()
        n, dev = graph.n_nodes, X.device
        n_loc = X.shape[0]
        ghost = dist.ghost if dist is not None else None
        H, D, LZ, Fp, Rp = geom.H, geom.D, geom.LZ, geom.Fp, geom.Rp
        f32 = dict(dtype=torch.float32, device=dev)
        dout = dout.contiguous()
        if ghost is not None:                               # + the owners' gradient rows of the split hub rows
            dout = _ghost_dout(ghost, dout, n_loc, n)
        dhn = torch.empty(n, H * D, **f32)
        dden = torch.empty(n, H, **f32)
        _lib.check(lib.spk_agg_bwd_pre(_lib.ptr(out), _lib.ptr(dout), out.stride(0), _lib.ptr(den), H, D,
                                       int(ctx.apply_elu), _lib.ptr(dhn), dhn.stride(0), _lib.ptr(dden), n,
                                       _lib.stream_ptr()), "agg_bwd_pre")
        dZ = torch.empty(n, H * LZ, **f32)
        dWa = torch.empty_like(Wa)
        for h in range(H):
            dh = dhn[:, h * D:(h + 1) * D]
            gemm_nn(dh, Wa[h].t().contiguous(), out=dZ[:, h * LZ:(h + 1) * LZ])
            if ghost is None:
                gemm_tn(Z[:, h * LZ:(h + 1) * LZ], dh, out=dWa[h])
            else:                                           # ghost rows are replicated: only their owner counts them
                gemm_tn(Z[:n_loc, h * LZ:(h + 1) * LZ], dh[:n_loc], out=dWa[h])
                gemm_tn((Z[n_loc:, h * LZ:(h + 1) * LZ] * ghost.mine.unsqueeze(1)).contiguous(), dh[n_loc:], out=dWa[h],
                        accumulate=True)
        Gx = torch.empty(n, _row_stride(H * Fp, GX_ALIGN), **f32)[:, :H * Fp]     # rows gathered per edge: stride rounded so
        Gr = torch.empty(n, _row_stride(H * Rp, GX_ALIGN), **f32)[:, :H * Rp]     # that a row does not straddle extra lines
        rowout = torch.empty(n, Fp + 4, **f32)
        a = _lib.AggBwdArgs()
        a.xrow = Xt.data_ptr(); a.ldxr = Xt.stride(0)
        a.dz = dZ.data_ptr(); a.ldz = dZ.stride(0)
        a.den = den.data_ptr(); a.sw = sw.data_ptr(); a.dden = dden.data_ptr()
        a.gx = Gx.data_ptr(); a.ldgx = Gx.stride(0); a.gr = Gr.data_ptr(); a.ldgr = Gr.stride(0)
        a.rowout = rowout.data_ptr(); a.ldro = rowout.stride(0)
        a.n_rows = n; a.alpha = float(ctx.alpha); a.geom = geom.struct()
        gx_geom, gr_geom = Geometry(H, Fp), Geometry(H, Rp)
        dXc = torch.empty(graph.n_cols, gx_geom.Wd, **f32)
        dRc = torch.empty(graph.n_rel, gr_geom.Wd, **f32)
        split = AGG_BWD_MODE == "split" and graph.t2 is None and Fp == Rp
        if split:
            # split-dot schedule (round 2): the per-edge dot t = c + Yb . x_j + Yc . r_k is formed in the two passes that
            # gather Gx[i] / Gr[i] anyway (column pass: x_j of the column in registers; relation pass: r_k in registers),
            # exactly as in the projected layer; the row-major pass that re-gathered X~[j] per edge is gone (2 row gathers
            # per edge in this backward instead of 3)
            rowsc = torch.empty(max(1, n), H, 4, **f32)
            a.rowsc = rowsc.data_ptr()
            _lib.check(lib.spk_agg_bwd_ctx(C.byref(a), _lib.stream_ptr()), "agg_bwd_ctx")
            del dZ
            ne = max(1, graph.n_edges)
            q = _lib.EdgeBwdSplitArgs()
            b = q.base
            b.rowptr = graph.rowptr.data_ptr()
            b.colptr = graph.colptr.data_ptr(); b.csc_row = graph.csc_row.data_ptr(); b.csc_pos = graph.csc_pos.data_ptr()
            b.csc_t1 = graph.csc_t1.data_ptr()
            b.P1 = Xc.data_ptr(); b.ld1 = Xc.stride(0)                      # (unused: the node pass is spk_agg_bwd_ctx)
            b.P2 = Xc.data_ptr(); b.ld2 = Xc.stride(0); b.P3 = Rt.data_ptr(); b.ld3 = Rt.stride(0)
            if ctx.mask_csr is not None:
                b.mask = ctx.mask_csr.data_ptr(); b.mask_stride = ctx.mask_csr.stride(0)
            b.G = Gx.data_ptr(); b.ldg = Gx.stride(0); b.rowsc = rowsc.data_ptr()
            b.dP1 = dXc.data_ptr(); b.ldd1 = dXc.stride(0)                  # (unused: the row sums go to `rowsum`)
            b.dP2 = dXc.data_ptr(); b.ldd2 = dXc.stride(0)
            b.n_rows = n; b.n_cols = graph.n_cols; b.apply_elu = 0; b.alpha = float(ctx.alpha)
            b.geom = gx_geom.struct()
            graph.row_hubs.fill(b.row_hub, None, 0)
            partc = _hub_partial(graph.col_hubs, gx_geom.Wd, dev)
            graph.col_hubs.fill(b.col_hub, partc, gx_geom.Wd)
            q.relptr = graph.relptr.data_ptr(); q.rel_row = graph.rel_row.data_ptr(); q.rel_pos = graph.rel_pos.data_ptr()
            rec4 = torch.empty(ne, H, 4, **f32); dsv = torch.empty(ne, H, **f32)
            q.rec4 = rec4.data_ptr(); q.dsv = dsv.data_ptr()
            q.dP3 = dRc.data_ptr(); q.ldd3 = dRc.stride(0); q.n_rel = graph.n_rel
            part3 = _hub_partial(graph.rel_hubs, gr_geom.Wd, dev)
            graph.rel_hubs.fill(q.rel_hub, part3, gr_geom.Wd)
            part1 = _hub_partial(graph.row_hubs, 4, dev)
            graph.row_hubs.fill(q.base.row_hub, part1, 4)
            rowsum = torch.empty(max(1, n), H, **f32)
            q.rowsum = rowsum.data_ptr(); q.ld_rowsum = H
            q.G_rel = Gr.data_ptr(); q.ldg_rel = Gr.stride(0)
            q.dup = 1

            def run(phases, tag):
                q.phases = phases
                _lib.current_tag = tag + f":w{gx_geom.Wd}"
                try:
                    _lib.check(lib.spk_edge_attn_bwd_split(C.byref(q), _lib.stream_ptr()), "edge_attn_bwd_split")
                finally:
                    _lib.current_tag = ""
        else:
            rec = torch.empty(max(1, graph.n_edges), 2 * H, **f32)
            a.segptr = graph.rowptr.data_ptr(); a.col = graph.col.data_ptr(); a.t1 = graph.t1.data_ptr()
            a.t2 = graph.t2.data_ptr() if graph.t2 is not None else None
            a.xcol = Xc.data_ptr(); a.ldxc = Xc.stride(0)
            a.rel = Rt.data_ptr(); a.ldr = Rt.stride(0)
            if ctx.mask_csr is not None:
                a.mask = ctx.mask_csr.data_ptr(); a.mask_stride = ctx.mask_csr.stride(0)
            rowsc = torch.empty(max(1, n), 8, **f32)                # (a rank may own no rows at all)
            a.rowsc = rowsc.data_ptr(); a.rec = rec.data_ptr()
            part = _hub_partial(graph.row_hubs, 8, dev)
            graph.row_hubs.fill(a.hub, part, 8)
            _lib.check(lib.spk_agg_bwd_rows(C.byref(a), _lib.stream_ptr()), "agg_bwd_rows")
            del dZ
        # column pass: dX through the gathered side, per head chunk; relation pass: dRel
        if split:
            run(2, "cols")
        else:
            seg_gather(graph.colptr, graph.csc_row, graph.csc_pos, graph.col_hubs, Gx, Gx.stride(0), rec, gx_geom, dXc,
                       graph.n_cols, "cols")
        if dist is not None:                              # partial sums over this rank's edges -> owners: the reduce-
            dXc_all = dXc                                 # scatter runs under the relation pass
            dXc_pad = torch.empty(dist.part.max_rows, gx_geom.Wd, **f32)
            hx = dist.reduce_scatter_start(dXc_all, dXc_pad)
        if split:
            run(4, "rels")                                # relation pass + row sums of ds
            rowout[:, Fp:Fp + H] = rowsum[:n]             # dq1 = sum of ds over the row
            # dq2 = sum of ds over the column (needs the relation pass): straight into the q slot of dXc on one GPU; with
            # the partial dXc already on its way to the owners, into a separate [n_cols, H] array reduce-scattered on its own
            if dist is not None:
                colsum = torch.empty(graph.n_cols, H, **f32)
                q.colsum = colsum.data_ptr(); q.ld_colsum = H
            run(8, "colsums")
            if dist is not None:
                qs_pad = torch.empty(dist.part.max_rows, H, **f32)
                hq = dist.reduce_scatter_start(colsum, qs_pad)
        else:
            seg_gather(graph.relptr, graph.rel_row, graph.rel_pos, graph.rel_hubs, Gr, Gr.stride(0), rec, gr_geom, dRc,
                       graph.n_rel, "rels")
        if dist is not None:
            dist.all_reduce(dRc)
            dist.all_reduce(dWa)
            if ghost is not None:                         # row-side gradient of a hub row = sum of the ranks' partials
                gsum = ghost.sum_partials(rowout[n_loc:].contiguous())
                rowout[ghost.mine_local] = gsum[ghost.mine]
            hx.wait()
            dXc = dXc_pad[:n_loc]
            del dXc_all
            if split:
                hq.wait()
                dXc[:, H * Fp:H * Fp + H].copy_(qs_pad[:n_loc])
        n = n_loc
        dX = torch.empty(n, geom.F, **f32)
        dq = torch.empty(n, 4, **f32)
        _lib.check(lib.spk_agg_dx(_lib.ptr(rowout), rowout.stride(0), _lib.ptr(dXc), dXc.stride(0), _lib.ptr(V), n,
                                  geom.F, geom.Fx4, H, _lib.ptr(dX), dX.stride(0), _lib.ptr(dq), _lib.stream_ptr()),
                   "agg_dx")
        dV = gemm_tn(Xt[:n, :geom.F], dq) if ctx.needs_input_grad[3] else None     # Xt rows start with x (16 B aligned stride)
        if dV is not None and dist is not None:
            dist.all_reduce(dV)
        dq3 = dRc[:, H * Rp:H * Rp + H].contiguous()                      # [R, H]
        dRel = None
        if ctx.needs_input_grad[1]:
            dRel = dRc[:, :geom.Rd].clone()
            for h in range(1, H):
                dRel += dRc[:, h * Rp:h * Rp + geom.Rd]
            dRel = gemm_nn(dq3, V3[:, :H].t().contiguous(), out=dRel, accumulate=True)
        dV3 = None
        if ctx.needs_input_grad[4]:
            dV3 = torch.zeros_like(V3)
            dV3[:, :H] = gemm_tn(Rel, dq3)
        return dX, dRel, dWa, dV, dV3, None, None, None, None, None, None


def attention_group(X, Rel, a_list, a2_list, graph, alpha, apply_elu, mask_csr, nanflag):
    """All heads of one layer (looping over groups of <=4): returns [N, sum_h D]."""
    outs = []
    # the C ABI takes raw pointers without row counts: check here what the reference's indexing would have caught
    # (IndexError from x[edge[..]] / relation_embed[edge_type], GAT/layers.py:129, models.py:156)
    if X.shape[0] != graph.n_nodes - getattr(graph, "n_ghost", 0):
        raise IndexError(f"entity table has {X.shape[0]} rows but the graph was built for "
                         f"{graph.n_nodes - getattr(graph, 'n_ghost', 0)} nodes")
    if getattr(graph, "dist", None) is None and graph.n_cols > X.shape[0]:
        raise IndexError(f"graph gathers from {graph.n_cols} nodes but the entity table has {X.shape[0]} rows")
    if Rel.shape[0] < graph.n_rel:
        raise IndexError(f"relation table has {Rel.shape[0]} rows but the graph uses {graph.n_rel} relations")
    if X.device != graph.device or Rel.device != graph.device:
        raise RuntimeError(f"tables on {X.device} / {Rel.device} but the graph layouts live on {graph.device}")
    F = X.shape[1]
    D = a_list[0].shape[0]
    Rd = a_list[0].shape[1] - 2 * F
    if use_agg_path(min(len(a_list), AGG_MAX_HEADS), F, Rd, D, graph):
        for g0 in range(0, len(a_list), AGG_MAX_HEADS):
            al, a2l = a_list[g0:g0 + AGG_MAX_HEADS], a2_list[g0:g0 + AGG_MAX_HEADS]
            geom = AggGeometry(len(al), F, Rd, D)
            Wa, V, V3 = agg_weights(al, a2l, geom)
            m = None if mask_csr is None else mask_csr[g0:g0 + AGG_MAX_HEADS].contiguous()
            outs.append(AggGroupFn.apply(X, Rel, Wa, V, V3, graph, geom, alpha, apply_elu, m, nanflag))
        return outs[0] if len(outs) == 1 else torch.cat(outs, dim=1)
    for g0 in range(0, len(a_list), MAX_HEADS):
        al, a2l = a_list[g0:g0 + MAX_HEADS], a2_list[g0:g0 + MAX_HEADS]
        geom = Geometry(len(al), D)
        Wn, Wr = extended_weights(al, a2l, F, geom)
        m = None if mask_csr is None else mask_csr[g0:g0 + MAX_HEADS].contiguous()
        out, _, _ = AttentionGroupFn.apply(X, Wn, Rel, Wr, graph, geom, alpha, apply_elu, m, nanflag)
        outs.append(out)
    return outs[0] if len(outs) == 1 else torch.cat(outs, dim=1)


# ---- row-wise wrappers -----------------------------------------------------------------------

def rownorm_(x):
    """In-place L2 row normalisation of a contiguous [N, F] tensor (models.py:160-161)."""
    assert x.dim() == 2 and x.stride(1) == 1
    _lib.check(_lib.load().spk_rownorm(_lib.ptr(x), x.stride(0), _lib.ptr(x), x.stride(0), x.shape[0], x.shape[1],
                                       _lib.stream_ptr()), "rownorm")
    return x


def rownorm(x):
    x = x.contiguous()
    y = torch.empty_like(x)
    _lib.check(_lib.load().spk_rownorm(_lib.ptr(x), x.stride(0), _lib.ptr(y), y.stride(0), x.shape[0], x.shape[1],
                                       _lib.stream_ptr()), "rownorm")
    return y


def mask_from_index(idx, n_rows, device, flag=None):
    """mask[unique(idx)] = 1 (models.py:167-173); duplicates are harmless so no unique() is needed. An index outside
    [-n_rows, n_rows) is the reference's IndexError: raised here for host tensors (checked on the host, no device sync);
    for device tensors the kernel ORs 2 into `flag` (the model's sticky flag word, read once per forward by check_nanflag),
    or, without `flag`, into a private word that is read back here."""
    mask = torch.zeros(n_rows, dtype=torch.float32, device=device)
    if idx.numel() and not idx.is_cuda:
        if int(idx.min()) < -n_rows or int(idx.max()) >= n_rows:
            raise IndexError("batch_entities index out of range")
    idx = idx.to(device=device, dtype=torch.int64).contiguous()
    if idx.numel():
        own = flag is None
        if own:
            flag = torch.zeros(1, dtype=torch.int32, device=device)
        _lib.check(_lib.load().spk_mask_from_index(_lib.ptr(idx), idx.numel(), _lib.ptr(mask), n_rows, _lib.ptr(flag),
                                                   _lib.stream_ptr()), "mask_from_index")
        if own and int(flag.item()) & 2:
            raise IndexError("batch_entities index out of range")
    return mask


class ResidualNormFn(torch.autograd.Function):
    """normalize(EW + mask[:,None]*x2) (models.py:175-179)."""

    @staticmethod
    def forward(ctx, EW, x2, mask):
        EW = EW.contiguous(); x2 = x2.contiguous()
        n, w = EW.shape
        out = torch.empty_like(EW)
        inv = torch.empty(n, dtype=torch.float32, device=EW.device)
        _lib.check(_lib.load().spk_residual_norm_fwd(_lib.ptr(EW), EW.stride(0), _lib.ptr(x2), x2.stride(0),
                                                     _lib.ptr(mask), _lib.ptr(out), out.stride(0), _lib.ptr(inv),
                                                     n, w, _lib.stream_ptr()), "residual_norm_fwd")
        ctx.save_for_backward(out, mask, inv)
        return out

    @staticmethod
    def backward(ctx, g):
        out, mask, inv = ctx.saved_tensors
        g = g.contiguous()
        n, w = out.shape
        dew = torch.empty_like(out)
        dx2 = torch.empty_like(out)
        _lib.check(_lib.load().spk_residual_norm_bwd(_lib.ptr(g), g.stride(0), _lib.ptr(out), out.stride(0),
                                                     _lib.ptr(mask), _lib.ptr(inv), _lib.ptr(dew), dew.stride(0),
                                                     _lib.ptr(dx2), dx2.stride(0), n, w, _lib.stream_ptr()),
                   "residual_norm_bwd")
        return dew, dx2, None


# ---- linear probe loss (SURVEY.md 8d: loss = <out_entity, G_e> + <out_relation, G_r>) ---------------------------------

class InnerProductFn(torch.autograd.Function):
    """sum_k <a_k, b_k> as a 0-dim tensor on the library's deterministic reduction (no library dot on the path)."""

    @staticmethod
    def forward(ctx, *tensors):
        k = len(tensors) // 2
        a_list = [t.contiguous() for t in tensors[:k]]
        b_list = [t.contiguous() for t in tensors[k:]]
        lib = _lib.load()
        dev = a_list[0].device
        out = torch.empty(1, dtype=torch.float32, device=dev)
        ws = torch.empty(lib.spk_inner_product_workspace_bytes(), dtype=torch.uint8, device=dev)
        for i, (a, b) in enumerate(zip(a_list, b_list)):
            assert a.shape == b.shape and a.dtype == b.dtype == torch.float32
            _lib.check(lib.spk_inner_product(_lib.ptr(a), _lib.ptr(b), a.numel(), _lib.ptr(ws), _lib.ptr(out), int(i > 0),
                                             _lib.stream_ptr()), "inner_product")
        ctx.save_for_backward(*a_list, *b_list)
        return out.reshape(())

    @staticmethod
    def backward(ctx, g):
        t = ctx.saved_tensors
        k = len(t) // 2
        grads = [g * t[k + i] if ctx.needs_input_grad[i] else None for i in range(k)]
        grads += [g * t[i] if ctx.needs_input_grad[k + i] else None for i in range(k)]
        return tuple(grads)


def inner_product(a_list, b_list):
    """sum_k <a_list[k], b_list[k]> (differentiable)."""
    return InnerProductFn.apply(*a_list, *b_list)


def linear_loss_backward(outs, grads):
    """loss = sum_k <outs[k], grads[k]> and its backward pass. d loss / d outs[k] IS grads[k], so the backward is seeded with
    the G tensors directly (what loss.backward() computes after multiplying them by 1.0); returns the detached loss."""
    with torch.no_grad():
        loss = inner_product([o.detach() for o in outs], list(grads))
    torch.autograd.backward(list(outs), [g.to(o.dtype) for o, g in zip(outs, grads)])
    return loss
