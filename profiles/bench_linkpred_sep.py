"""Timing of the GAT_sep_space filtered link-prediction evaluation (recon_b200.entity_ranks with model_gat) on one B200:
CUDA events, inputs resident. Prints one JSON line.
  python profiles/bench_linkpred_sep.py [--reps 3] [--ab-groups 64]
Workload: that of profiles/bench_linkpred.py (N = 2M entities, D = 200, R = 1000, 20M known triples from synth.make_kg,
T = 1000 test rows drawn from the known set, both sides) plus a seeded xavier-uniform W_ent2rel [R, D, D] (160 MB). The
rows fall into one group per distinct relation, most of 1-3 rows; each group costs two [N, D] x [D, *] GEMMs (tanh(E W_r)
and AC_r = P_r [W1a^T | W1c^T]) and one count + filter per side. The [N, 2D] table (3.2 GB) is far larger than the
126 MB L2, so every count pass streams it from HBM.
Reported:
  * whole_call_ms: the median of --reps calls, each ending in its own host synchronisation;
  * phase_ms: per-entry-point CUDA events in a separate pass, summed over the relations (tanh GEMM, AC GEMM, count and
    filter per side);
  * count_tile_ab: the count phase of the first --ab-groups relation groups, each group once as it is (narrow pair
    tiles) and once padded to 128 rows with keep = 0 (the 128-row tile), same candidate table, per side;
  * count_tile_crossover: count time for n pairs (n = 16 .. 128) as ceil(n / 16) calls of at most 16 rows (narrow
    tiles) against one call padded to 128 rows (128-row tile); the narrow-tile threshold of spk_linkpred_count
    (LP_NARROW_MAX) is read off it;
  * oracle: ranks of a seeded sample of 64 rows against the fp64 vectorised sep-space oracle
    (tests/linkpred_sep_oracle.py), every difference required to be a near tie (|s_c - s_true| <= 1e-5 max(1, |s_true|)).
"""
import argparse
import json
import os
import subprocess
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))                            # the sep-space oracle
import torch  # noqa: E402

from bench_linkpred import _model, _smi  # noqa: E402


def _events():
    return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


def _timed(fn, reps=3):
    """Median CUDA-event time of fn() in ms over reps runs after one warm-up."""
    fn()
    out = []
    for _ in range(reps):
        e0, e1 = _events()
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1))
    return sorted(out)[len(out) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--ab-groups", type=int, default=64)
    args = ap.parse_args()
    from recon_b200 import KnownTriples, entity_ranks, _lib
    from recon_b200 import functional as SF
    from recon_b200.linkpred import _head_weights
    from recon_b200.convkb import LRELU_SLOPE
    from recon_b200.synth import make_kg
    import linkpred_sep_oracle as S
    dev = torch.device("cuda:0")
    torch.manual_seed(0)                                                   # the ConvKB layers' default init
    n, d, r_n, m, t_n = 2_000_000, 200, 1000, 20_000_000, 1000
    gen = torch.Generator(device=dev).manual_seed(0)
    edge, etype, _ = make_kg(n, m, r_n, alpha=1.1, seed=0, device=dev, hub_frac=0.5)
    known_tri = torch.stack((edge[1], etype, edge[0]), 1).contiguous()
    del edge, etype
    tri = known_tri[torch.randint(0, m, (t_n,), device=dev, generator=gen)].contiguous()
    model = _model(n, d, r_n, dev, gen)
    bound = (6.0 / (2 * d)) ** 0.5                                        # xavier_uniform of a [D, D] matrix
    w = (torch.rand(r_n, d, d, device=dev, generator=gen) * 2 - 1) * bound
    gat = types.SimpleNamespace(W_ent2rel=w)
    known = KnownTriples(known_tri, n, r_n)
    del known_tri
    sizes = torch.bincount(tri[:, 1], minlength=r_n)
    present = sizes.nonzero().flatten()
    hist = torch.bincount(sizes[present]).tolist()
    group_hist = {str(k): v for k, v in enumerate(hist) if v}

    rh, rt = entity_ranks(model, tri, known, model_gat=gat)              # warm-up
    try:                                                                   # SM clock samples while the timed calls run
        clock = subprocess.Popen(["nvidia-smi", "--query-gpu=clocks.sm", "--format=csv,noheader,nounits", "-i", "0",
                                  "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
    except OSError:
        clock = None
    times = []
    for _ in range(args.reps):
        e0, e1 = _events()
        e0.record()
        rh2, rt2 = entity_ranks(model, tri, known, model_gat=gat)
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    clocks = []
    if clock is not None:
        clock.terminate()
        clocks = [int(x) for x in clock.communicate()[0].split() if x.strip().isdigit()]
    same_twice = bool(torch.equal(rh, rh2) and torch.equal(rt, rt2))
    whole = sorted(times)[len(times) // 2]
    print(f"whole call: {times} ms over {int(present.numel())} relations", file=sys.stderr, flush=True)

    # per-phase CUDA events: gemm tags are "MxKxN"; count / filter alternate head, tail within a relation
    lib = _lib.load()
    lib.timing = []
    entity_ranks(model, tri, known, model_gat=gat)
    torch.cuda.synchronize()
    phase, seen = {}, {}
    for name, a, b in lib.timing:
        base, _, tag = name.partition(":")
        if base.startswith("gemm"):
            mm, _, nn = tag.split("x")
            key = "gemm_bt" if int(mm) != n else ("gemm_tanh_p" if int(nn) == d else "gemm_ac")
        elif base.startswith("linkpred"):
            k = seen.get(base, 0)
            seen[base] = k + 1
            key = f"{base}_{'head' if k % 2 == 0 else 'tail'}"
        else:
            key = base
        phase[key] = phase.get(key, 0.0) + a.elapsed_time(b)
    lib.timing = None
    n_rel_present = int(present.numel())

    # count-phase A/B on the real groups: narrow tiles (the group as it is) against the 128-row tile (padded, keep = 0)
    w_ac, bt, b1, w2 = _head_weights(model)
    ent = SF.tc_friendly(model.final_entity_embeddings.detach().contiguous())
    p_buf = torch.empty(n, d, device=dev)
    ac = torch.empty(n, 2 * d, device=dev)
    err = torch.zeros(1, dtype=torch.int32, device=dev)
    order = torch.sort(tri[:, 1], stable=True).indices
    tri_s = tri[order].contiguous()
    offs = torch.cumsum(sizes, 0) - sizes
    v = torch.empty(128, d, device=dev)
    st = torch.empty(128, device=dev)
    tid = torch.empty(128, dtype=torch.int32, device=dev)
    cnt = torch.empty(128, dtype=torch.int32, device=dev)

    def count(rows, keep, side):
        _lib.check(lib.spk_linkpred_count(_lib.ptr(ac), ac.stride(0), n, _lib.ptr(bt), bt.stride(0), r_n, _lib.ptr(b1),
                                          _lib.ptr(w2), LRELU_SLOPE, d, _lib.ptr(rows), _lib.ptr(keep),
                                          rows.shape[0], side, _lib.ptr(v), d, _lib.ptr(st), _lib.ptr(tid),
                                          _lib.ptr(cnt), _lib.ptr(err), _lib.stream_ptr()), "linkpred_count")

    ab = {"narrow_ms": [0.0, 0.0], "tile128_ms": [0.0, 0.0], "groups": 0, "rows": 0}
    for r in present[:args.ab_groups].tolist():
        c, lo = int(sizes[r]), int(offs[r])
        SF.gemm_nn(ent, w[r], out=p_buf, act=2)
        SF.gemm_nn(p_buf, w_ac, out=ac)
        rows = tri_s[lo:lo + c].contiguous()
        padded = torch.cat((rows, rows[:1].expand(128 - c, 3)), 0).contiguous() if c < 128 else rows
        keep_pad = (torch.arange(padded.shape[0], device=dev) < c).to(torch.uint8)
        for side in (0, 1):
            ab["narrow_ms"][side] += _timed(lambda: count(rows, None, side))
            ab["tile128_ms"][side] += _timed(lambda: count(padded, keep_pad, side))
        ab["groups"] += 1
        ab["rows"] += c
    ab["speedup"] = sum(ab["tile128_ms"]) / sum(ab["narrow_ms"])
    print(f"phases: {phase}\ncount A/B: {ab}", file=sys.stderr, flush=True)

    # crossover: n pairs as ceil(n / 16) narrow calls against one 128-row tile (same table: the last relation's)
    cross = []
    for k in (16, 32, 48, 64, 80, 96, 112, 128):
        rows = tri[:k].contiguous()
        keep_pad = torch.ones(128, dtype=torch.uint8, device=dev)
        keep_pad[k:] = 0
        padded = torch.cat((rows, tri[:128 - k]), 0).contiguous()

        def narrow():
            for i in range(0, k, 16):
                count(rows[i:i + 16], None, 1)
        cross.append({"pairs": k, "narrow16_ms": _timed(narrow), "tile128_ms": _timed(lambda: count(padded, keep_pad, 1))})
    print(f"crossover: {cross}", file=sys.stderr, flush=True)
    del p_buf, ac

    # oracle on a seeded sample of 64 rows
    gs = torch.Generator().manual_seed(1)
    sample = torch.randperm(t_n, generator=gs)[:64]
    p = {"final_entity_embeddings": model.final_entity_embeddings.detach(),
         "final_relation_embeddings": model.final_relation_embeddings.detach(),
         "convKB.fc1.weight": model.convKB.fc1.weight.detach(), "convKB.fc1.bias": model.convKB.fc1.bias.detach(),
         "convKB.fc2.weight": model.convKB.fc2.weight.detach(), "convKB.fc2.bias": model.convKB.fc2.bias.detach()}
    kn = torch.stack(((known.tail_keys // n) // r_n, (known.tail_keys // n) % r_n, known.tail_keys % n), 1)
    fh, ft, nh, nt = S.filtered_ranks(p, tri[sample.to(dev)], kn, n, w, device=dev)
    sh, st_ = rh[sample], rt[sample]
    oracle = {"rows": 64, "exact_head": int((sh == fh).sum()), "exact_tail": int((st_ == ft).sum()),
              "all_differences_near_ties": bool(((sh - fh).abs() <= nh).all() and ((st_ - ft).abs() <= nt).all())}

    mhz = sorted(clocks)[len(clocks) // 2] if clocks else None
    res = {"workload": f"linkpred GAT_sep_space: N={n} D={d} R={r_n} known={m} T={t_n} (both sides, all rows evaluated)",
           "gpu": torch.cuda.get_device_name(0), "power_limit": _smi("power.limit"),
           "sm_clock_mhz_median_during_timed_calls": mhz,
           "sm_clock_mhz_range": [min(clocks), max(clocks)] if clocks else None,
           "relations_present": n_rel_present, "group_size_histogram": group_hist,
           "whole_call_ms_median": whole, "whole_call_ms": times, "ms_per_relation": whole / n_rel_present,
           "phase_ms": phase, "phase_ms_per_relation": {k: v / n_rel_present for k, v in phase.items()},
           "count_tile_ab": ab, "count_tile_crossover": cross, "oracle": oracle,
           "rank_head_mean": float(rh.double().mean()), "rank_tail_mean": float(rt.double().mean()),
           "bit_identical_repeat": same_twice}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
