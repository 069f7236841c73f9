"""Timing of the filtered link-prediction evaluation (recon_b200.entity_ranks) on one B200: CUDA events, inputs resident.
Workload: N = 2M entities, D = 200, R = 1000, 20M known triples from synth.make_kg (head = edge[1], tail = edge[0]: Zipf
tails, so (., r, t) hub ranges occur), T = 1000 test rows drawn from the known set; every row is evaluated on both sides.
The [N, 2D] candidate table (3.2 GB) and the 20M-key arrays are far larger than the 126 MB L2. Prints one JSON line.
  python profiles/bench_linkpred.py [--reps 5] [--no-ab]
Phases (per-entry-point CUDA events, a separate pass): the [A | C] and Bt GEMMs, spk_linkpred_count and
spk_linkpred_filter per side; the whole call is timed without per-phase events and ends in its own host sync.
Work: 2 T N (pair, candidate) scores of D elements each. The count kernel's inner loop issues FP32_INSTR_PER_ELEMENT
instructions per element: FADD (x = a + v), FMUL (slope * x), FMNMX (lrelu = max(x, slope * x)), FFMA (acc += w2 * lrelu),
read from `cuobjdump -sass` of lp_count_kernel (1024 of each per unrolled 8 x 64 x 8 step pair, nothing else on FP32).
fp32_issue_share = elements * FP32_INSTR_PER_ELEMENT / (count-kernel time * SMs * 128 lanes * observed SM clock).
A/B in the same run: the same ranks from the existing spk_rank_scores (the T x N score matrix, 8 GB per side), with the
known candidates masked and the count done by torch; rows whose ranks differ can only be near ties (different sum order).
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

FP32_INSTR_PER_ELEMENT = 4


def _smi(query):
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={query}", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30)
        return out.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return "unavailable"


def _model(n, d, r, dev, gen):
    from recon_b200 import SpKBGATConvOnly
    m = SpKBGATConvOnly(torch.zeros(1, 4), torch.zeros(1, 4), [d, d], [d, d], 0.0, 0.0, 0.2, 0.2, [1, 1], 1).to(dev)
    m.final_entity_embeddings = torch.nn.Parameter(torch.randn(n, d, device=dev, generator=gen))
    m.final_relation_embeddings = torch.nn.Parameter(torch.randn(r, d, device=dev, generator=gen))
    return m


def _ab_ranks(model, tri, known):
    """Ranks through the materialised score matrix: spk_rank_scores per side, known candidates set to -inf, torch count."""
    from recon_b200 import _lib
    from recon_b200.convkb import LRELU_SLOPE
    from recon_b200.linkpred import _score_tables
    lib = _lib.load()
    n, r_n = known.n_entities, known.n_relations
    ac, bt, b1, w2 = _score_tables(model)
    d = bt.shape[1]
    b2 = model.convKB.fc2.bias.detach().contiguous()
    h, r, t = tri[:, 0], tri[:, 1], tri[:, 2]
    t_n = tri.shape[0]
    out, near = [], []
    for side, keys in ((0, known.head_keys), (1, known.tail_keys)):
        x = ac[:, :d] if side == 0 else ac[:, d:2 * d]
        v = (((ac[t, d:2 * d] if side == 0 else ac[h, :d]) + bt[r]) + b1).contiguous()
        true = h if side == 0 else t
        s = torch.empty(t_n, n, dtype=torch.float32, device=tri.device)
        _lib.check(lib.spk_rank_scores(_lib.ptr(v), v.stride(0), _lib.ptr(x), x.stride(0), _lib.ptr(w2), _lib.ptr(b2),
                                       LRELU_SLOPE, t_n, n, d, _lib.ptr(s), s.stride(0), _lib.stream_ptr()), "rank_scores")
        st = s.gather(1, true.unsqueeze(1))
        base = ((t if side == 0 else h) * r_n + r) * n
        lo = torch.searchsorted(keys, base)
        lens = torch.searchsorted(keys, base + n) - lo
        rows = torch.repeat_interleave(torch.arange(t_n, device=tri.device), lens)
        start = torch.cumsum(lens, 0) - lens
        pos = lo[rows] + torch.arange(rows.numel(), device=tri.device) - start[rows]
        cand = keys[pos] - base[rows]
        other = cand != true[rows]
        s[rows[other], cand[other]] = float("-inf")                       # repeated keys: the same cell twice
        gt = (s > st) | (torch.isnan(s) & ~torch.isnan(st))
        out.append(gt.sum(1) + 1)
        near.append(((s - st).abs() <= 1e-5 * st.abs().clamp(min=1.0)).sum(1) - 1)
        del s, gt
    return out, near


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--no-ab", action="store_true")
    args = ap.parse_args()
    from recon_b200 import KnownTriples, entity_ranks, _lib
    from recon_b200.synth import make_kg
    dev = torch.device("cuda:0")
    n, d, r_n, m, t_n = 2_000_000, 200, 1000, 20_000_000, 1000
    gen = torch.Generator(device=dev).manual_seed(0)
    edge, etype, _ = make_kg(n, m, r_n, alpha=1.1, seed=0, device=dev, hub_frac=0.5)
    known_tri = torch.stack((edge[1], etype, edge[0]), 1).contiguous()
    del edge, etype
    tri = known_tri[torch.randint(0, m, (t_n,), device=dev, generator=gen)].contiguous()
    model = _model(n, d, r_n, dev, gen)

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    known = KnownTriples(known_tri, n, r_n)
    e1.record()
    torch.cuda.synchronize()
    known_ms = e0.elapsed_time(e1)

    rh, rt = entity_ranks(model, tri, known)                               # warm-up (module load, GEMM set-up)
    try:                                                                   # SM clock samples while the timed calls run
        clock = subprocess.Popen(["nvidia-smi", "--query-gpu=clocks.sm", "--format=csv,noheader,nounits", "-i", "0",
                                  "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
    except OSError:
        clock = None
    times = []
    for _ in range(args.reps):
        e0.record()
        rh2, rt2 = entity_ranks(model, tri, known)
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    clocks = []
    if clock is not None:
        clock.terminate()
        clocks = [int(x) for x in clock.communicate()[0].split() if x.strip().isdigit()]
    same_twice = bool(torch.equal(rh, rh2) and torch.equal(rt, rt2))

    lib = _lib.load()
    phases = {}
    for _ in range(args.reps):
        lib.timing = []
        entity_ranks(model, tri, known)
        torch.cuda.synchronize()
        seen, rep = {}, {}
        for name, a, b in lib.timing:
            base = name.split(":")[0]
            k = seen.get(base, 0)
            seen[base] = k + 1
            key = "gemm_prologue" if base.startswith("gemm") else f"{base}_{'head' if k == 0 else 'tail'}"
            rep[key] = rep.get(key, 0.0) + a.elapsed_time(b)
        for key, ms in rep.items():
            phases.setdefault(key, []).append(ms)
        lib.timing = None
    phase_ms = {k: sum(v) / len(v) for k, v in phases.items()}

    whole = sorted(times)[len(times) // 2]
    elems = 2 * t_n * n * d
    count_ms = phase_ms.get("linkpred_count_head", 0.0) + phase_ms.get("linkpred_count_tail", 0.0)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    mhz = sorted(clocks)[len(clocks) // 2] if clocks else None
    res = {"workload": f"linkpred: N={n} D={d} R={r_n} known={m} T={t_n} (both sides, all rows evaluated)",
           "gpu": torch.cuda.get_device_name(0), "power_limit": _smi("power.limit"),
           "sm_clock_mhz_median_during_timed_calls": mhz, "sm_clock_mhz_range": [min(clocks), max(clocks)] if clocks else None,
           "known_triples_build_ms": known_ms, "whole_call_ms_median": whole, "whole_call_ms": times,
           "phase_ms": phase_ms, "pair_candidates_per_s": 2 * t_n * n / (whole * 1e-3),
           "elements_per_s": elems / (whole * 1e-3), "count_kernel_elements_per_s": elems / (count_ms * 1e-3),
           "fp32_instr_per_element": FP32_INSTR_PER_ELEMENT,
           "fp32_issue_share_count_kernel": (elems * FP32_INSTR_PER_ELEMENT / (count_ms * 1e-3 * sms * 128 * mhz * 1e6)
                                             if mhz else None),
           "rank_head_mean": float(rh.double().mean()), "rank_tail_mean": float(rt.double().mean()),
           "bit_identical_repeat": same_twice}
    if not args.no_ab:
        with torch.no_grad():
            _ab_ranks(model, tri, known)                                   # warm-up
            e0.record()
            (ah, at), (nh, nt) = _ab_ranks(model, tri, known)
            e1.record()
            torch.cuda.synchronize()
        ab_ms = e0.elapsed_time(e1)
        dh, dt = (ah.cpu() != rh), (at.cpu() != rt)
        res.update({"ab_score_matrix_ms": ab_ms, "ab_speedup": ab_ms / whole,
                    "ab_rows_differing_head": int(dh.sum()), "ab_rows_differing_tail": int(dt.sum()),
                    "ab_differing_rows_all_near_ties": bool(((ah.cpu() - rh).abs() <= nh.cpu()).all()
                                                            and ((at.cpu() - rt).abs() <= nt.cpu()).all())})
    print(json.dumps(res))


if __name__ == "__main__":
    main()
