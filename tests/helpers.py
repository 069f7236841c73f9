"""Shared helpers for the parity tests."""
import os
import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

MODEL_CASES = ["model_small_uniform", "model_small_zipf_nhop", "model_small_dropmask",
               "model_refdims", "model_batch_test", "model_3heads"]


def load_golden(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    return {k: z[k] for k in z.files}


def rel_l2(a, b):
    def _t(x):
        if isinstance(x, torch.Tensor):
            return x.detach().cpu().double().flatten()
        return torch.as_tensor(np.asarray(x)).double().flatten()
    a, b = _t(a), _t(b)
    den = b.norm().item()
    return (a - b).norm().item() / (den if den > 0 else 1.0)


# ---- the GEMM dispatch, restated (spk_gemm_tc.cu gemm_nn_tc / tn_plan, spk_gemm_simt.cu, functional.gemm_nn / gemm_tn) --
B200_SMS = 148                    # SM count the GEMM's grids and pair / cluster thresholds are computed from on a B200
TC_BM, TC_BK = 128, 32            # tcgen05 M tile and k-block (one 128 B swizzle row of fp32)
TC_SMEM = 225 * 1024 - 1024       # dynamic shared memory the pipeline ring and the epilogue staging may use
SIMT_BAND = 65535 * 128           # rows of one gemm_nn_simt launch (grid.y <= 65535 tiles of 128 rows)


def tc_nn_plan(m, n, k, c_vec, accumulate=False, act=0, path="tc", sms=B200_SMS):
    """Plan of spk_gemm_tc.cu gemm_nn_tc (and of gemm_nn_tc_grouped, which copies its tile shape, epilogue and depth) for
    C[m, n] (+)= A[m, k] B[k, n]; c_vec = C's row stride and base both allow 16-byte stores. `path` "tc-pair" / "tc-cluster"
    is SPK_TC_PAIR=1 / SPK_TC_CLUSTER=2. tiles_per_cta is the most work items one persistent CTA runs (for clusters and
    pairs assuming every SM can host one: the launch asks the occupancy API)."""
    n_tiles_n = (n + 255) // 256
    bn_round = 32 if n_tiles_n > 1 else 16          # several N tiles: whole 32-column store boxes per tile
    bn = max(16, -(-(-(-n // n_tiles_n)) // bn_round) * bn_round)
    c_tma = bool(c_vec and n % 4 == 0 and not (act and accumulate))
    staging = 4 * 8192 if c_tma else 0
    m_tiles = -(-m // TC_BM)
    big = m_tiles * n_tiles_n >= 2 * sms
    if path == "tc-pair" and c_tma and bn % 16 == 0 and big:
        kernel, stage_bytes = "pair", 2 * TC_BM * TC_BK * 4 + bn * 128
        items, ctas_per_item = -(-m_tiles // 2) * n_tiles_n, 2
    else:
        kernel = "cluster" if path == "tc-cluster" and not accumulate and big else "tc"
        stage_bytes = 2 * TC_BM * TC_BK * 4 + 2 * bn * 128
        ctas_per_item = 2 if kernel == "cluster" else 1
        items = -(-m_tiles // ctas_per_item) * n_tiles_n
    stages = min(4, (TC_SMEM - staging) // stage_bytes)
    per_cta = -(-items // min(items, sms // ctas_per_item))
    return dict(kernel=kernel, n_tiles_n=n_tiles_n, BN=bn, stages=stages,
                epilogue="tma" if c_tma else "row-vec4" if c_vec else "row-scalar",
                num_kb=-(-k // TC_BK), m_tiles=m_tiles, tiles_per_cta=per_cta)


def gemm_nn_branch(m, n, lda, ldc, accumulate, act, path, sms=B200_SMS):
    """(kernel, epilogue) of functional.gemm_nn(act=act) for a 16-byte aligned A / C allocation: the SIMT GEMM followed by
    spk_elu_inplace, or spk_gemm_tc.cu gemm_nn_tc (TMA-store epilogue when c_vec && !(act && accumulate), else the
    per-thread-row epilogue, float4 when C allows it), its pair-CTA kernel (SPK_TC_PAIR=1) or 2-CTA clusters
    (SPK_TC_CLUSTER=2), both only once there are 2 x sms tiles of 128 rows. TMA stores only whole rows of 16-byte
    units, so N % 4 != 0 takes the per-thread-row epilogue. BN is always a multiple of 16 and the raw tile is the hi
    operand by default, so the pair kernel's other conditions always hold."""
    if path == "simt" or n > 512 or lda % 4:
        return "simt", "elu_inplace"
    pl = tc_nn_plan(m, n, 1, ldc % 4 == 0, accumulate, act, path, sms)
    return pl["kernel"], pl["epilogue"]


def tc_tn_plan(m, ka, nb):
    """spk_gemm_tc.cu tn_plan: one CTA per (Ka tile of 128, Nb tile of BN, m split); splits of whole 32-row stages."""
    p = dict(n_tiles_k=-(-ka // 128), n_tiles_n=-(-nb // 256))
    p["BN"] = -(-(-(-nb // p["n_tiles_n"])) // 32) * 32
    splits = max(1, min(-(-B200_SMS // (p["n_tiles_k"] * p["n_tiles_n"])), -(-m // 1024)))
    mps = max(32, -(-(-(-m // splits)) // 32) * 32)
    p["splits"], p["m_per_split"] = -(-m // mps), mps
    p["last_split_rows"] = m - (p["splits"] - 1) * mps
    p["stages"] = max(1, min(4, TC_SMEM // ((4 + p["BN"] // 32) * 4096) - 2))
    return p


def simt_nn_bands(m):
    """spk_gemm_simt.cu gemm_nn_simt: launches of at most 65535 row tiles."""
    return -(-m // SIMT_BAND)


def simt_tn_splits(m, ka, nb):
    """spk_gemm_simt.cu gemm_tn_splits: ~8 CTAs of 64 x 64 per SM, at least 1024 rows per split, at most 512 splits."""
    tiles = -(-ka // 64) * -(-nb // 64)
    return max(1, min(512, -(-B200_SMS * 8 // tiles), -(-m // 1024)))


def golden_params(g, dtype=torch.float32):
    return {k[len("param."):]: torch.as_tensor(v).to(dtype) for k, v in g.items() if k.startswith("param.")}


def golden_masks(g, dtype=torch.float32):
    m = {k[len("mask."):]: torch.as_tensor(v).to(dtype) for k, v in g.items() if k.startswith("mask.")}
    return m or None
