"""Timing of the GAT_sep_space TransE loss (recon_b200.loss.batch_gat_loss with model_gat) on one B200: CUDA events,
inputs resident. Writes profiles/loss_sep_bench.json (or --out) and prints it as one JSON line.
  python profiles/bench_loss_sep.py [--reps 5] [--pos 2000,20000,100000] [--out PATH]
Workload: N = 2M entities, HD = 200, R = 1000 relations drawn with Zipf(1.1) frequencies, ratio 2, P positives (T = 5P
rows: P positives, then P head- and P tail-corrupted negatives per ratio step), so the projection sees 2T = 10P rows.
The entity table (1.6 GB) is far larger than the 126 MB L2.
Reported per P:
  * loss_fwd_bwd_ms: median of --reps calls of loss forward + backward (the loss's own error check synchronises);
  * kernels: per-entry-point CUDA events of one more call (a separate pass): the grouped forward GEMM (Y = tanh(X W_r)),
    the grouped dX GEMM, the grouped dW GEMM with its fixed-order reduce, their algorithmic TFLOP/s at 2 * 2T * HD^2
    each (pad rows not counted), and the layout kernels;
  * pad_share: pad rows / padded rows of that batch; launches_per_call: spk_launch_count over one loss forward + backward;
  * projection_ab: the relation-space projection of the 2T rows, forward + backward, by the grouped path
    (convkb.ent2rel_project) and by the per-relation loop of the previous release (kept below as _loop_project),
    alternated in the same run; at the smallest P also the reference's eager torch form (bmm over a gathered
    [2T, HD, HD] copy of W_ent2rel).
Card name, power limit and the median SM clock sampled during the timed calls are recorded beside the numbers.
"""
import argparse
import json
import os
import subprocess
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402


def _smi(query):
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={query}", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30)
        return out.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return "unavailable"


def _median_ms(fn, reps):
    fn()
    out = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1))
    return sorted(out)[len(out) // 2]


class _LoopMatMulFn(torch.autograd.Function):
    """The previous release's grouped product: one tensor-core GEMM per relation present, host-side offsets."""

    @staticmethod
    def forward(ctx, Xs, W, rel_sorted_ids, offsets):
        from recon_b200 import functional as SF
        Xs = SF.tc_friendly(Xs.contiguous())
        d_out = W.shape[2]
        Y = torch.empty(Xs.shape[0], (d_out + 3) // 4 * 4, dtype=torch.float32, device=Xs.device)[:, :d_out]
        for r, lo, hi in zip(rel_sorted_ids, offsets[:-1], offsets[1:]):
            SF.gemm_nn(Xs[lo:hi], W[r], out=Y[lo:hi])
        ctx.save_for_backward(Xs, W)
        ctx.seg = (rel_sorted_ids, offsets)
        return Y

    @staticmethod
    def backward(ctx, g):
        from recon_b200 import functional as SF
        Xs, W = ctx.saved_tensors
        rel_ids, offsets = ctx.seg
        g = SF.tc_friendly(g.contiguous())
        dX = torch.empty(Xs.shape[0], (Xs.shape[1] + 3) // 4 * 4, dtype=torch.float32, device=Xs.device)[:, :Xs.shape[1]]
        dW = torch.zeros_like(W)
        for r, lo, hi in zip(rel_ids, offsets[:-1], offsets[1:]):
            SF.gemm_nn(g[lo:hi], W[r].t().contiguous(), out=dX[lo:hi])
            SF.gemm_tn(Xs[lo:hi], g[lo:hi], out=dW[r])
        return dX, dW, None, None


def _loop_project(rows, w_ent2rel, rel_ids):
    """The previous release's ent2rel_project (bincount().tolist() on the host, one GEMM per relation and pass)."""
    from recon_b200.convkb import GatherRowsFn, TanhFn
    order = torch.sort(rel_ids, stable=True).indices
    counts = torch.bincount(rel_ids, minlength=w_ent2rel.shape[0]).tolist()
    present = [r for r, c in enumerate(counts) if c]
    offsets = [0]
    for r in present:
        offsets.append(offsets[-1] + counts[r])
    xs = GatherRowsFn.apply(rows, order)
    ys = TanhFn.apply(_LoopMatMulFn.apply(xs, w_ent2rel, present, offsets))
    inv = torch.empty_like(order)
    inv[order] = torch.arange(order.numel(), device=order.device)
    return GatherRowsFn.apply(ys, inv)


def _eager_project(rows, w_ent2rel, rel_ids):
    """The reference's form (GAT_sep_space/main.py:360-377): bmm against a gathered [rows, HD, HD] copy of W_ent2rel."""
    return torch.tanh(torch.bmm(rows.unsqueeze(1), w_ent2rel[rel_ids]).squeeze(1))


def _batch(n_ent, n_rel, n_pos, ratio, gen, dev):
    ranks = torch.arange(1, n_rel + 1, dtype=torch.float64)
    prob = ranks.pow(-1.1)
    rel = torch.multinomial(prob / prob.sum(), n_pos, replacement=True, generator=gen)
    pos = torch.stack((torch.randint(0, n_ent, (n_pos,), generator=gen), rel,
                       torch.randint(0, n_ent, (n_pos,), generator=gen)), dim=1)
    neg = pos.repeat(2 * ratio, 1)
    half = ratio * n_pos
    neg[:half, 0] = torch.randint(0, n_ent, (half,), generator=gen)
    neg[half:, 2] = torch.randint(0, n_ent, (half,), generator=gen)
    return torch.cat((pos, neg), dim=0).to(dev)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--pos", default="2000,20000,100000")
    ap.add_argument("--n-ent", type=int, default=2_000_000)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "loss_sep_bench.json"))
    args = ap.parse_args()
    from recon_b200 import _lib
    from recon_b200.convkb import RelationLayout, ent2rel_project
    from recon_b200.loss import batch_gat_loss
    if not torch.cuda.is_available():
        raise SystemExit("bench_loss_sep.py needs a CUDA device")
    dev = torch.device("cuda:0")
    lib = _lib.load()
    n_ent, hd, n_rel, ratio = args.n_ent, 200, 1000, 2
    gen = torch.Generator().manual_seed(0)
    ent = torch.randn(n_ent, hd, generator=gen).to(dev).requires_grad_(True)
    rel = torch.randn(n_rel, hd, generator=gen).to(dev).requires_grad_(True)
    w = (torch.randn(n_rel, hd, hd, generator=gen) / hd ** 0.5).to(dev).requires_grad_(True)
    gat = types.SimpleNamespace(W_ent2rel=w)
    f = torch.nn.MarginRankingLoss(margin=5.0)

    try:                                                                   # SM clock samples while the timed calls run
        clock = subprocess.Popen(["nvidia-smi", "--query-gpu=clocks.sm", "--format=csv,noheader,nounits", "-i", "0",
                                  "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
    except OSError:
        clock = None

    results = []
    for n_pos in [int(x) for x in args.pos.split(",")]:
        tri = _batch(n_ent, n_rel, n_pos, ratio, gen, dev)
        t = tri.shape[0]

        def loss_step():
            for p in (ent, rel, w):
                p.grad = None
            batch_gat_loss(f, tri, ent, rel, valid_invalid_ratio_gat=ratio, model_gat=gat).backward()

        loss_ms = _median_ms(loss_step, args.reps)
        torch.cuda.synchronize()
        c0 = lib.spk_launch_count()
        loss_step()
        torch.cuda.synchronize()
        launches = lib.spk_launch_count() - c0
        lib.timing = []
        loss_step()
        torch.cuda.synchronize()
        per = {}
        nn_calls = 0
        for name, e0, e1 in lib.timing:
            if name == "gemm_nn_tc_grouped":
                name = "gemm_nn_tc_grouped:" + ("forward_tanh" if nn_calls == 0 else "dX")
                nn_calls += 1
            per[name] = per.get(name, 0.0) + e0.elapsed_time(e1)
        lib.timing = None
        flops = 2.0 * (2 * t) * hd * hd
        kernels = {k: {"ms": round(v, 4)} for k, v in sorted(per.items())}
        for k in ("gemm_nn_tc_grouped:forward_tanh", "gemm_nn_tc_grouped:dX", "gemm_tn_tc_grouped"):
            if k in kernels:
                kernels[k]["algorithmic_tflops"] = round(flops / (per[k] * 1e-3) / 1e12, 1)
        lay = RelationLayout(tri[:, 1], t, 2, 3, n_rel)
        n_groups, n_tiles, n_tasks = lay.counts.tolist()
        pad_share = 1.0 - (2 * t) / (128.0 * n_tiles)

        # projection A/B: grouped path against the per-relation loop, alternated; the same 2T gathered rows
        ids = torch.cat((tri[:, 0], tri[:, 2]))
        rid = torch.cat((tri[:, 1], tri[:, 1]))
        rows = ent.detach()[ids].contiguous().requires_grad_(True)
        gy = torch.randn(rows.shape[0], hd, generator=gen).to(dev)

        def proj(fn):
            def run():
                rows.grad = None
                w.grad = None
                (fn(rows, w, rid) * gy).sum().backward()
            return run

        ab = {"grouped_ms": [], "loop_ms": []}
        for _ in range(3):
            ab["grouped_ms"].append(round(_median_ms(proj(ent2rel_project), args.reps), 3))
            ab["loop_ms"].append(round(_median_ms(proj(_loop_project), args.reps), 3))
        with torch.no_grad():
            y_new, y_old = ent2rel_project(rows, w, rid), _loop_project(rows, w, rid)
            ab["max_abs_diff_outputs"] = float((y_new - y_old).abs().max())
        g_med, l_med = sorted(ab["grouped_ms"])[1], sorted(ab["loop_ms"])[1]
        ab["speedup_over_loop"] = round(l_med / g_med, 2)
        if n_pos == min(int(x) for x in args.pos.split(",")):
            ab["eager_torch_ms"] = round(_median_ms(proj(_eager_project), args.reps), 3)
            ab["speedup_over_eager"] = round(ab["eager_torch_ms"] / g_med, 2)
        results.append({"P": n_pos, "T": t, "projected_rows": 2 * t, "relations_present": n_groups,
                        "m_tiles": n_tiles, "dw_tasks": n_tasks, "pad_share": round(pad_share, 4),
                        "loss_fwd_bwd_ms": round(loss_ms, 3), "launches_per_call": int(launches),
                        "kernels": kernels, "projection_ab": ab})
        del tri, rows, gy, lay
        torch.cuda.empty_cache()

    clocks = []
    if clock is not None:
        clock.terminate()
        clocks = [int(x) for x in clock.communicate()[0].split() if x.strip().isdigit()]
    out = {"bench": "loss_sep", "gpu": torch.cuda.get_device_name(0), "power_limit": _smi("power.limit"),
           "sm_clock_max": _smi("clocks.max.sm"),
           "sm_clock_mhz_median_during_run": sorted(clocks)[len(clocks) // 2] if clocks else None,
           "n_ent": n_ent, "hd": hd, "n_rel": n_rel, "zipf": 1.1, "ratio": ratio, "reps": args.reps,
           "results": results}
    line = json.dumps(out)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        fh.write(json.dumps(out, indent=1) + "\n")
    print(line)


if __name__ == "__main__":
    main()
