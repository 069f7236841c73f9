"""bench.py -- SpKBGAT fwd+bwd edges/sec on synthetic power-law KGs (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c2|c1|c3|c4|c5] [--impl reference]
                  [--dump-outputs DIR]

A step = SpKBGATModified forward (2 attention layers) + loss.backward() over the whole graph, loss =
<out_entity, G_e> + <out_relation, G_r> (SURVEY.md 8d), batch_entities = arange(N) (dense mask).
`value`   : edges/s with the graph layouts and all inputs resident in HBM.
`e2e`     : edges/s through the public module call with HOST edge tensors: every step copies the pinned
            int64 edge list / types / 2-hop rows to the device, rebuilds CSR+CSC+relation layouts on the
            device, runs fwd+bwd and reads the loss back.
`roofline`: the dominant kernel's algorithmic bytes / its CUDA-event time, against MEASURED_PEAKS.json.
`cpu_baseline`: the CPU port of the reference path (oracle/ref_torch.py, COO sparse.sum like the reference)
            on a bounded sample, host cores of this box.
--dump-outputs DIR writes what the last timed step handed to its caller (outputs, loss, parameter gradients) as
            DIR/<name>.npy; inputs are seeded, so two builds run with the same arguments can be compared array by array.
The benchmark writes nothing into the source tree (it may be read-only).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True        # no __pycache__ in the source tree
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

WORKLOADS = {
    # name: (N, E1, E2, R, zipf_alpha, hub_frac)   hub_frac: share of edges whose row is Pareto-distributed
    "c1": (10_000, 100_000, 0, 200, 1.1, 1.0),
    "c2": (2_000_000, 20_000_000, 0, 1_000, 1.1, 0.2),
    "c3": (2_000_000, 20_000_000, 40_000_000, 1_000, 1.1, 0.2),
    "c4": (20_000_000, 400_000_000, 0, 2_000, 1.1, 0.2),
    "c5": (5_000_000, 100_000_000, 0, 1_000, 1.1, 1.0),
}
F_IN, D_OUT, HEADS, ALPHA = 50, 100, 2, 0.2


def b_alg_bytes(n, e1, e2):
    """BASELINE.md section 5: B_layer = E(12 Dt + 24 + 16 H + 8[2hop]) + N(48 Dt + 8 F), two layers."""
    dt = D_OUT * HEADS
    def layer(f_in, h):
        return (e1 + e2) * (12 * dt + 24 + 16 * h) + 8 * e2 + n * (48 * dt + 8 * f_in)
    return layer(F_IN, HEADS) + layer(dt, 1)


def make_inputs(name, seed=0, device="cpu"):
    from recon_b200.synth import make_kg
    n, e1, e2, r, alpha, hub_frac = WORKLOADS[name]
    edge, etype, nhop = make_kg(n, e1, r, alpha, e2, seed, device=device, hub_frac=hub_frac)
    return n, r, edge, etype, nhop


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower() == "active"})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


def cpu_reference_arm(steps, warmup, threads=None, one_thread=True):
    """The reference's own CPU implementation on the C1 sample: the UNMODIFIED /root/reference/GAT/{layers,models}.py
    (copied by build() into the git-ignored oracle/_ref/, module globals CUDA pinned to False: SURVEY.md 8c/8d) through
    its public module call; falls back to the oracle port (kind "port") only when oracle/_ref was never installed."""
    from oracle import ref_loader
    from recon_b200.synth import make_kg
    n, e1, e2, r, alpha, _ = WORKLOADS["c1"]
    edge, etype, nhop = make_kg(n, e1, r, alpha, e2, 0)
    g = torch.Generator().manual_seed(1)
    ge, gr = torch.randn(n, D_OUT * HEADS, generator=g), torch.randn(r, D_OUT * HEADS, generator=g)
    be = torch.arange(n)
    ref = ref_loader.load()
    if ref is not None:
        kind = "reference"
        g0 = torch.Generator().manual_seed(0)
        ent, rel = torch.randn(n, F_IN, generator=g0), torch.randn(r, F_IN, generator=g0)
        torch.manual_seed(0)
        model = ref[1].SpKBGATModified(ent, rel, [D_OUT, 2 * D_OUT], [D_OUT, 2 * D_OUT], 0.0, ALPHA, [HEADS, HEADS], None)

        def step():
            model.zero_grad()
            out_e, out_r, _ = model(None, be, (edge, etype), nhop)
            ((out_e * ge).sum() + (out_r * gr).sum()).backward()
    else:
        kind = "port"
        from oracle import ref_torch as O
        p = O.init_params(n, r, F_IN, D_OUT, HEADS, seed=0)

        def step():
            O.fwd_bwd(p, be, (edge, etype), nhop, ALPHA, ge, gr)

    def timed(nthreads, k, w):
        torch.set_num_threads(nthreads)
        ts = []
        for i in range(w + k):
            t0 = time.perf_counter()
            step()
            if i >= w:
                ts.append(time.perf_counter() - t0)
        ts.sort()
        return ts[len(ts) // 2]

    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        cores = threads or os.cpu_count()
        med = timed(cores, steps, warmup)
        med1 = timed(1, 2, 1) if one_thread else None
        torch.set_num_threads(cores)
    out = {"value": (e1 + e2) / med, "unit": "edges/s", "cores": cores, "kind": kind,
           "sample": f"C1 shape N={n} E={e1} R={r} Zipf {alpha} (largest the reference algorithm holds: it "
                     f"materialises [2F+Rd,E]); median of {steps} fwd+bwd after {warmup} warm-ups, fp32, dropout off",
           "ms_per_step": med * 1e3}
    if med1 is not None:
        out["one_thread"] = {"value": (e1 + e2) / med1, "unit": "edges/s", "cores": 1, "ms_per_step": med1 * 1e3}
    return out


def add_workload(name):
    """c2xK: K x the C2 shape (weak-scaling family); c4h: half of C4 in both N and E (the largest power-of-two fraction
    of the 400M-edge scale-out shape whose single-GPU step fits 180 GB: C4 itself needs ~220 GB on one GPU)."""
    if name in WORKLOADS:
        return
    if name.startswith("c5/"):        # C5's shape divided by k (same Pareto(1.1) rows: the top row still holds ~53 % of the edges)
        k = int(name[3:])
        n0, e0, _, r0, a0, h0 = WORKLOADS["c5"]
        WORKLOADS[name] = (n0 // k, e0 // k, 0, r0, a0, h0)
    elif name.startswith("c2x"):
        k = int(name[3:])
        n0, e0, _, r0, a0, h0 = WORKLOADS["c2"]
        WORKLOADS[name] = (n0 * k, e0 * k, 0, r0, a0, h0)
    elif name == "c4h":
        n0, e0, _, r0, a0, h0 = WORKLOADS["c4"]
        WORKLOADS[name] = (n0 // 2, e0 // 2, 0, r0, a0, h0)
    else:
        raise SystemExit(f"unknown workload {name}")


def describe(workload):
    n_, e1_, e2_, r_, a_, h_ = WORKLOADS[workload]
    return (f"{workload}: N={n_} E1={e1_} E2={e2_} R={r_} in={F_IN} entity_out=[{D_OUT},{2 * D_OUT}] "
            f"heads=[{HEADS},{HEADS}] rows: {int(100 * h_)}% Pareto(alpha={a_}) hubs + uniform")


def run_config(workload, world, rank, dev, steps, warmup, want_prof=False, want_e2e=False, clocks=False, dump_dir=None):
    """Builds the runner for `workload`, runs `warmup` untimed + `steps` timed steps (CUDA events, barrier + synchronize on
    both sides, max over ranks). With `dump_dir`, what the last timed step computed is written there (dump_outputs) before
    anything else runs. Returns a dict; the runner is released before returning."""
    import torch.distributed as dist
    from recon_b200 import _lib, profiler
    add_workload(workload)
    n, r, edge, etype, nhop = make_inputs(workload, device=dev if (world > 1 or WORKLOADS[workload][1] > 50_000_000) else "cpu")
    e_total = edge.shape[1] + nhop.shape[0]
    if world > 1:
        from recon_b200.dist import PartitionedKBGAT
        runner = PartitionedKBGAT(n, r, edge, etype, nhop, F_IN, D_OUT, HEADS, ALPHA, dev)
    else:
        runner = SingleGPU(n, r, edge, etype, nhop, dev)
    del edge, etype, nhop
    torch.cuda.empty_cache()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(warmup):
        runner.step()
    barrier()
    sampler = ClockSampler(dev.index or 0) if (clocks and rank == 0) else None
    if sampler:
        sampler.start()
    torch.cuda.reset_peak_memory_stats()
    l0 = _lib.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(steps):
        runner.keep_outputs = dump_dir is not None and i == steps - 1
        runner.step()
    ev1.record()
    barrier()
    res = {"workload": workload, "e_total": e_total, "launches": _lib.launch_count() - l0,
           "peak_mem_gb": round(torch.cuda.max_memory_allocated() / 2 ** 30, 1)}
    if dump_dir is not None:
        res["dump"] = dump_outputs(runner, dump_dir)
    ms = ev0.elapsed_time(ev1) / steps
    res["clocks"] = sampler.stop() if sampler else None
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        lo = torch.tensor([runner.n_edges_local], device=dev, dtype=torch.float64)
        hi = lo.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN); dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        res["edges_per_rank"] = {"min": int(lo.item()), "max": int(hi.item())}
    res["ms"] = ms
    if want_prof:                     # per-call timing pass (CUDA events around every C-ABI call on the launching stream)
        prof_steps = max(2, min(steps, 5))
        profiler.enable()
        for _ in range(prof_steps):
            runner.step()
        res["prof"], res["prof_steps"] = profiler.disable(), prof_steps
        if world == 1:
            res["graph_build_ms"] = runner.graph_build_ms()
    if want_e2e and world == 1:
        res["e2e"] = runner.e2e(max(2, min(steps, 5)))
        res["e2e_pipelined"] = runner.e2e_pipelined(max(2, min(steps, 5)))
    elif want_e2e:
        sec, h2d = runner.e2e(max(2, min(steps, 3)))
        t = torch.tensor([sec, float(h2d)], device=dev, dtype=torch.float64)
        tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        res["e2e"] = {"value": e_total / float(tmax[0]), "unit": "edges/s", "h2d_bytes_per_step": int(tsum[1]),
                      "d2h_bytes_per_step": 4 * world, "ms_per_step": float(tmax[0]) * 1e3,
                      "includes": "per rank: pinned H2D of its int64 edge list, device CSR/CSC/relation build, fwd+bwd "
                                  "with the exchanges, loss D2H; max over ranks"}
    if world == 1 and want_prof:
        res["runner_roofline"] = runner.roofline
        res["roofline_args"] = (res["prof"],)
        peaks = {}
        pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(pk):
            peaks = json.load(open(pk))
        hbm_peak, peak_src = (peaks["hbm_gbs"], "measured") if "hbm_gbs" in peaks else (6650.0, "fallback")
        res["roofline"] = runner.roofline(res["prof"], hbm_peak, peak_src)
        res["hbm_peak"], res["peak_src"] = hbm_peak, peak_src
        del res["runner_roofline"], res["roofline_args"]
    del runner
    import gc
    gc.collect()
    torch.cuda.empty_cache()
    return res


DUMP_ROWS = 32768                    # entity rows kept per entity-indexed array: ~33 MB at the default widths
DUMP_LIMIT = 64 * 2 ** 20


def dump_outputs(runner, out_dir):
    """Writes what the runner's last step returned to its caller -- out_entity, out_relation, mask, the loss and the
    gradient of every parameter -- as out_dir/<name>.npy in float32 (float64 for float64 tensors). Arrays indexed by entity
    are cut to the same fixed, seeded sample of DUMP_ROWS rows, stored as `sample_rows`."""
    import numpy as np
    out = dict(runner.outputs)
    for name, prm in runner.model.named_parameters():
        if prm.grad is not None:
            out["grad." + name] = prm.grad
    n = runner.n
    rows = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:DUMP_ROWS].sort().values
    arrays = {"sample_rows": rows.double()}
    rows = rows.to(runner.dev)
    for k, v in out.items():
        v = v.detach()
        if k in ("out_entity", "mask", "grad.entity_embeddings"):
            v = v.index_select(0, rows)
        arrays[k] = v.cpu().to(torch.float64 if v.dtype == torch.float64 else torch.float32)
    total = sum(a.numel() * a.element_size() for a in arrays.values())
    if total > DUMP_LIMIT:
        raise RuntimeError(f"output dump of {total} bytes exceeds {DUMP_LIMIT}")
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a.numpy())
    return {"dir": out_dir, "arrays": len(arrays), "bytes": total}


def config_of(workload, world):
    """`config` of the JSON line; the reference arm prints the same object (it runs a bounded sample of this workload)."""
    return {"workload": describe(workload),
            "l2": "gather tables (P2 1.7 GB/layer) exceed the 126 MB L2; no flush needed",
            "parallelism": f"row-partition x{world}" if world > 1 else "single GPU"}


def secondary(res, world):
    """Compact record of a secondary measurement (strong-scaling shapes) for the JSON line."""
    n_, e1_, e2_, *_ = WORKLOADS[res["workload"]]
    balg = b_alg_bytes(n_, e1_, e2_)
    out = {"workload": describe(res["workload"]), "n_gpus": world, "ms_per_step": res["ms"],
           "value": res["e_total"] / (res["ms"] * 1e-3), "unit": "edges/s", "scaling": "strong",
           "frac_of_8TBs_per_gpu": balg / (res["ms"] * 1e-3) / 8e12 / world, "peak_mem_gb": res["peak_mem_gb"]}
    if "edges_per_rank" in res:
        out["edges_per_rank"] = res["edges_per_rank"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default=None)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-strong", action="store_true", help="skip the secondary strong-scaling shapes (c4h, c4)")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--sub", action="store_true", help="(internal) secondary measurement in a child process")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (one GPU, --impl ours)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.dump_outputs is not None and (world > 1 or args.gpus > 1 or args.impl != "ours"):
        ap.error("--dump-outputs needs the single-GPU path (--gpus 1, --impl ours)")
    # Primary line: the C2 shape per GPU (BASELINE configs[1] at N=1; N GPUs run N x 2M entities / N x 20M edges, row-
    # partitioned: weak scaling, so the driver's per-N efficiency is well defined). Secondary keys carry BASELINE
    # configs[3] (C4, 400M edges; N >= 4) and its half c4h (fits one GPU) as STRONG-scaling measurements at every N.
    default_mode = args.workload is None
    workload = args.workload or ("c2" if max(world, args.gpus) == 1 else f"c2x{max(world, args.gpus)}")
    add_workload(workload)

    if args.impl == "reference":
        if rank != 0:
            return
        base = cpu_reference_arm(args.steps, args.warmup)
        line = {"impl": "reference", "metric": "SpKBGAT fwd+bwd edges/sec", "value": base["value"], "unit": "edges/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": base["ms_per_step"],
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": config_of(workload, args.gpus),
                "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample", "one_thread") if k in base},
                "e2e": {"value": base["value"], "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    if args.sub:                       # child of a 1-GPU run: one secondary shape, compact line
        res = run_config(workload, world, rank, dev, args.steps, args.warmup)
        print("SUB " + json.dumps(secondary(res, world)))
        return

    res = run_config(workload, world, rank, dev, args.steps, args.warmup, want_prof=True, want_e2e=not args.no_e2e,
                     clocks=True, dump_dir=args.dump_outputs)
    if "dump" in res:
        print("[bench] outputs of the last timed step: " + json.dumps(res["dump"]), file=sys.stderr, flush=True)
    ms, e_total = res["ms"], res["e_total"]
    line = None
    if rank == 0:
        hbm_peak, peak_src = res.get("hbm_peak"), res.get("peak_src")
        if hbm_peak is None:
            pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
            peaks = json.load(open(pk)) if os.path.exists(pk) else {}
            hbm_peak, peak_src = (peaks["hbm_gbs"], "measured") if "hbm_gbs" in peaks else (6650.0, "fallback")
        n_, e1_, e2_, *_ = WORKLOADS[workload]
        balg = b_alg_bytes(n_, e1_, e2_)
        prof, prof_steps = res["prof"], res["prof_steps"]
        line = {"metric": "SpKBGAT fwd+bwd edges/sec", "value": e_total / (ms * 1e-3), "unit": "edges/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
                "scaling": "weak" if (world == 1 or workload.startswith("c2x")) else "strong", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": config_of(workload, world),
                "clocks": res["clocks"], "gpu_launches": res["launches"], "peak_mem_gb": res["peak_mem_gb"],
                "step_roofline": {"b_alg_bytes": balg, "achieved_gbs": balg / (ms * 1e-3) / 1e9 / world,
                                  "frac_of_8TBs": balg / (ms * 1e-3) / 8e12 / world,
                                  "frac_of_measured": balg / (ms * 1e-3) / (hbm_peak * 1e9) / world,
                                  "peak_source": peak_src, "per": "GPU"},
                "kernels_ms_per_step": {k: round(v[0] / prof_steps, 4) for k, v in sorted(prof.items(), key=lambda kv: -kv[1][0])}}
        for k in ("roofline", "e2e", "e2e_pipelined", "graph_build_ms", "edges_per_rank"):
            if res.get(k):
                line[k] = res[k]

    # ---- secondary sections; a watchdog prints what exists if one of them stalls (e.g. a rank out of memory inside a
    # collective), so the primary measurement is never lost ----
    import threading

    def bail():
        if rank == 0 and line is not None:
            line.setdefault("notes", []).append("secondary section timed out; primary line printed by the watchdog")
            print(json.dumps(line), flush=True)
        os._exit(0)

    dog = threading.Timer(420.0, bail)
    dog.daemon = True
    dog.start()
    if default_mode and not args.no_strong:
        shapes = ["c4h"] + (["c4"] if world >= 4 else [])
        for w in shapes:
            try:
                if world == 1:        # child process: an out-of-memory C4 attempt cannot take the primary line with it
                    if rank == 0:
                        p = subprocess.run([sys.executable, os.path.abspath(__file__), "--workload", w, "--steps", "3",
                                            "--warmup", "2", "--sub"], capture_output=True, text=True, timeout=300)
                        sub = [l for l in p.stdout.splitlines() if l.startswith("SUB ")]
                        line[w] = json.loads(sub[-1][4:]) if sub else {"error": (p.stderr or p.stdout)[-300:]}
                else:
                    r2 = run_config(w, world, rank, dev, 3, 2)
                    if rank == 0:
                        line[w] = secondary(r2, world)
                        print("[bench] " + w + ": " + json.dumps(line[w]), file=sys.stderr, flush=True)
            except Exception as exc:                 # noqa: BLE001
                if rank == 0:
                    line[w] = {"error": repr(exc)[:300]}
                if world > 1:
                    raise
    if rank == 0:
        print("[bench] primary: " + json.dumps({k: line[k] for k in ("value", "ms_per_step", "n_gpus")}), file=sys.stderr, flush=True)
    if world > 1 and not args.no_parity:
        from recon_b200.dist import parity_check
        try:
            par = parity_check(dev)
        except Exception as exc:                     # noqa: BLE001  (a failing rank leaves the others in a collective:
            par = {"error": repr(exc)[:300]}         #  the watchdog above then prints the line)
            if rank == 0:
                line["parity"] = par
                print(json.dumps(line), flush=True)
            os._exit(0 if rank == 0 else 1)
        if rank == 0:
            line["parity"] = par
    if rank == 0 and not args.no_cpu_baseline and world == 1:
        base = cpu_reference_arm(3, 1)
        line["cpu_baseline"] = {k: base[k] for k in ("value", "unit", "cores", "kind", "sample", "one_thread") if k in base}
    dog.cancel()
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


class SingleGPU:
    def __init__(self, n, r, edge, etype, nhop, dev):
        from recon_b200 import SpKBGATModified
        torch.manual_seed(0)
        self.dev, self.n, self.r = dev, n, r
        g = torch.Generator().manual_seed(0)
        ent = torch.randn(n, F_IN, generator=g)
        rel = torch.randn(r, F_IN, generator=g)
        self.model = SpKBGATModified(ent, rel, [D_OUT, 2 * D_OUT], [D_OUT, 2 * D_OUT], 0.0, ALPHA, [HEADS, HEADS], None).to(dev)
        self.edge, self.etype, self.nhop = edge.to(dev), etype.to(dev), nhop.to(dev)
        self._host = None if edge.is_cuda else (edge.pin_memory(), etype.pin_memory(), nhop.pin_memory())
        self.batch = torch.arange(n, device=dev)
        self.g_ent = torch.randn(n, D_OUT * HEADS, generator=g).to(dev)
        self.g_rel = torch.randn(r, D_OUT * HEADS, generator=g).to(dev)
        self.graph = self.model.prepare_graph((self.edge, self.etype), self.nhop)
        self.e = edge.shape[1] + nhop.shape[0]
        self.e1, self.e2 = edge.shape[1], nhop.shape[0]
        self.keep_outputs, self.outputs = False, None

    def step(self, graph=None, adj=None, nhop=None):
        """graph: prebuilt layouts (device-timed `value`); adj / nhop: the reference's call with HOST edge tensors (`e2e`).
        With `keep_outputs` set, what the step returns to its caller stays in `outputs` (the gradients stay in the model)."""
        self.model.zero_grad(set_to_none=True)
        if adj is not None:
            out_e, out_r, mask = self.model(None, self.batch, adj, nhop)
        else:
            out_e, out_r, mask = self.model(None, self.batch, graph or self.graph, None)
        # <out_entity, G_e> + <out_relation, G_r>  (SURVEY.md 8d) as two dot products
        # (the library's deterministic reduction for the value; the backward is seeded with G_e / G_r, which is d loss / d out)
        from recon_b200 import functional as SF
        loss = SF.linear_loss_backward((out_e, out_r), (self.g_ent, self.g_rel))
        if self.keep_outputs:
            self.outputs = {"out_entity": out_e.detach(), "out_relation": out_r.detach(), "mask": mask, "loss": loss}
        return loss

    @property
    def host(self):
        """Pinned host copies of the int64 edge tensors (the form the reference's data pipeline hands over)."""
        if self._host is None:
            self._host = tuple(t.cpu().pin_memory() for t in (self.edge, self.etype, self.nhop))
        return self._host

    def graph_build_ms(self, reps=3):
        """CSR + CSC + relation layouts from the device-resident int64 edge tensors (per graph, amortised over epochs;
        SURVEY.md 8d asks for it separately): CUDA events, mean of `reps` builds after one warm-up."""
        from recon_b200 import KGraph
        nh = self.nhop if self.nhop.numel() else None
        KGraph(self.edge, self.etype, nh, self.n, self.r, device=self.dev)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(reps):
            KGraph(self.edge, self.etype, nh, self.n, self.r, device=self.dev)
        ev1.record()
        torch.cuda.synchronize()
        return ev0.elapsed_time(ev1) / reps

    def e2e(self, steps):
        """One step through the public call with HOST int64 edge tensors, as the reference's training loop holds them:
        KGraph packs them to int32 in pinned memory (all host cores), copies them on a copy stream while the CSR / CSC /
        relation layouts are being built, then forward + backward + loss read-back. Nothing is cached between steps."""
        from recon_b200 import KGraph
        h_edge, h_type, h_nhop = self.host
        n_arr = 4 if h_nhop.numel() else 3
        h2d = 4 * n_arr * self.e                      # bytes that actually cross PCIe (int32 staging of the int64 tensors)
        res = torch.empty(1, dtype=torch.float32).pin_memory()
        times = []
        # the call a user of the reference makes: model(Corpus_, batch, (edge_list, edge_type), nhop) with the host tensors;
        # graph_cache off, so every step packs, copies and rebuilds the layouts (nothing is reused between steps)
        cache, self.model.graph_cache = self.model.graph_cache, False
        try:
            for i in range(steps + 1):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                loss = self.step(adj=(h_edge, h_type), nhop=h_nhop if h_nhop.numel() else None)
                res.copy_(loss.detach().reshape(1), non_blocking=True)
                torch.cuda.synchronize()
                if i > 0:
                    times.append(time.perf_counter() - t0)
        finally:
            self.model.graph_cache = cache
        t = sum(times) / len(times)
        return {"value": self.e / t, "unit": "edges/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                "ms_per_step": t * 1e3,
                "includes": "host pack of the int64 edge tensors to pinned int32 (all cores), H2D on a copy stream overlapped "
                            "with the device CSR/CSC/relation build, fwd+bwd, loss D2H",
                "host_int64_bytes_per_step": 8 * (3 * self.e1 + 4 * self.e2)}

    def e2e_pipelined(self, steps):
        """Same work and bytes per step as e2e(), but the pinned H2D copy of the NEXT step's edge tensors is issued on a
        copy stream at the start of each step (double buffering, what an input pipeline does), so it overlaps the
        device work. Extra information next to the strict `e2e`; never raises (returns {"error": ...})."""
        try:
            from recon_b200 import KGraph
            h_edge, h_type, h_nhop = self.host
            main = torch.cuda.current_stream()
            copy_stream = torch.cuda.Stream(device=self.dev)
            res = torch.empty(1, dtype=torch.float32).pin_memory()

            def prefetch():
                with torch.cuda.stream(copy_stream):
                    bufs = [h.to(self.dev, non_blocking=True) for h in (h_edge, h_type, h_nhop)]
                    ev = torch.cuda.Event()
                    ev.record(copy_stream)
                return bufs, ev

            nxt = prefetch()
            times = []
            for i in range(steps + 1):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                (edge, et, nh), ev = nxt
                main.wait_event(ev)
                for b in (edge, et, nh):
                    b.record_stream(main)
                nxt = prefetch()                       # one H2D of the full edge list per step, overlapped
                graph = KGraph(edge, et, nh if nh.numel() else None, self.n, self.r, device=self.dev)
                loss = self.step(graph)
                res.copy_(loss.detach().reshape(1), non_blocking=True)
                torch.cuda.synchronize()
                if i > 0:
                    times.append(time.perf_counter() - t0)
                del graph, edge, et, nh
            t = sum(times) / len(times)
            return {"value": self.e / t, "unit": "edges/s", "ms_per_step": t * 1e3,
                    "includes": "as e2e, with the H2D of the next step's edge tensors double-buffered on a copy stream"}
        except Exception as exc:                       # informational only: must not cost the bench line
            return {"error": repr(exc)[:200]}

    def roofline(self, prof, hbm_peak, peak_src):
        """Dominant edge kernel (largest share of the step) against the HBM peak. Algorithmic bytes per launch
        follow SURVEY.md 8d: per edge a 4*Dt-byte row gather + 8 B of indices (+8H record bytes in the backward
        passes, H averaged over the two layers), per node the Dt-wide rows each pass reads/writes."""
        dt = D_OUT * HEADS
        n, e = self.n, self.e
        h_avg = (HEADS + 1) / 2.0
        algs = {
            # K2: per edge the P2~[j] row (4 Dt) + col / type indices (8) (+4 per 2-hop edge); per node P1~ read + out write
            "edge_attn_fwd": e * (4 * dt + 8) + 4 * self.e2 + n * (8 * dt),
            "edge_attn_bwd_rows": e * (4 * dt + 8 + 8 * h_avg) + 4 * self.e2 + n * (20 * dt),
            "edge_attn_bwd_segments:cols": e * (4 * dt + 8 + 8 * h_avg) + n * (4 * dt),
            # split-dot backward of the projected layer (layer 2, H = 1), one gather kernel per timed call:
            #   column pass  = SURVEY 8d "pass B": per edge the dnum[i] row (4 Dt) + row index + position (8) + its record
            #                  (8 H); per column the P2~[j] read and the dP2~[j] write (8 Dt)
            #   relation pass: per edge the dnum[i] row again (4 Dt) + indices (8) + record (8 H); dP3~ is cache resident
            #   node pass    : per node dOut, out read and dnum, dP1~ written (16 Dt)
            "edge_attn_bwd_split:cols": e * (4 * dt + 8 + 8 * 1) + n * (8 * dt),
            "edge_attn_bwd_split:rels": e * (4 * dt + 8 + 8 * 1),
            "edge_attn_bwd_split:node": n * (16 * dt),
            "edge_attn_bwd_split": e * (8 * dt + 16 + 16 * 1) + n * (24 * dt),
        }
        cand = {}
        wd_proj = (dt + HEADS + 7) // 8 * 8          # table width of the projected path (208); narrower launches belong to
        for k, v in prof.items():                  # the aggregate-then-project layer and move fewer bytes than B_alg charges
            base, _, wtag = k.partition(":w") if ":w" in k else (k, "", "")
            if wtag and int(wtag) != wd_proj:
                continue
            if base in algs:
                ms0, c0 = cand.get(base, (0.0, 0))
                cand[base] = (ms0 + v[0], c0 + v[1])
        if not cand:
            return None
        top = max(cand, key=lambda k: cand[k][0])
        ms_launch = cand[top][0] / cand[top][1]
        achieved = algs[top] / (ms_launch * 1e-3) / 1e9
        traffic = None                         # dram__bytes_read+write per launch from the committed ncu capture (profiles/)
        tj = os.path.join(ROOT, "profiles", "r2_traffic.json")
        if os.path.exists(tj):
            traffic = json.load(open(tj)).get(f"c2:{top}") if (self.n, self.e) == (2_000_000, 20_000_000) else None
        cuda_kernels = {"edge_attn_fwd": "edge_fwd_stream_kernel<2,1,0,*> (rows + hub tasks) + edge_fwd_hub_finalize_kernel",
                        "edge_attn_bwd_split:cols": "split_cols_kernel<2,1,4,4> (+ split_cols_tasks_kernel for hub columns)",
                        "edge_attn_bwd_split:rels": "split_rels_tasks_kernel<2,1,4,4> (+ split_rels_kernel) + split_sum_kernel (rows)",
                        "edge_attn_bwd_split:node": "bwd_node_kernel<2,1>"}
        return {"bound": "hbm", "kernel": top, "cuda_kernels": cuda_kernels.get(top, top), "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                "frac": achieved / hbm_peak, "traffic": traffic, "peak_source": peak_src, "ms_per_launch": ms_launch,
                "alg_bytes_per_launch": algs[top],
                "all": {k: {"ms_per_launch": cand[k][0] / cand[k][1], "gbs": algs[k] / (cand[k][0] / cand[k][1] * 1e-3) / 1e9}
                        for k in cand}}


if __name__ == "__main__":
    main()
