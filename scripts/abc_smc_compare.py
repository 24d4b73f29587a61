"""ABC-SMC against rejection ABC on the C4 shape (1e5-cell birth-death runs, b1 ~ U(1, 2), d0, d1 ~ U(0, 0.5), the
target one run at (1.4, 0.2, 0.2), thresholds 0.05/0.1/0.1/0.1 times each of --scales), one GPU.  Writes
<out>/abc_smc_compare.json, per threshold scale:

- rejection ABC: draws and device time until the M-th accepted draw (or the acceptance rate over --rejection-max);
- ABC-SMC with population M: per generation epsilon, consumed and simulated draws, ESS, and the host-clock time of
  the simulation, proposal and weight steps;
- the weight kernel alone at N = M = --pairs-n: call time (host clock around the blocking call, copies included) and
  kernel time (torch.profiler, a run of its own), pair evaluations per second.

The card's name and power limit are read in the same run.  Usage: python scripts/abc_smc_compare.py OUT_DIR"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

THR = (0.05, 0.1, 0.1, 0.1)
BOX = dict(b1_range=(1.0, 2.0), d0_range=(0.0, 0.5), d1_range=(0.0, 0.5))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power, clock = (q.stdout.strip().split(", ") + ["not read"] * 3)[:3]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def valid_rho(dist, stop, thr):
    """rho = max_j d_j / thr_j over the enabled distances; inf for a draw ABC-SMC never accepts."""
    rho = np.zeros(len(dist), dtype=np.float32)
    with np.errstate(divide="ignore", invalid="ignore"):
        for j, t in enumerate(np.float32(thr)):
            if t >= 0:
                d = dist[:, j]
                r = np.where(d == 0, np.float32(0), np.float32(np.inf)) if t == 0 else (d / t).astype(np.float32)
                rho = np.maximum(rho, np.where(np.isnan(d), np.float32(np.inf), r))
    bad = ((stop & 0xFF) == 5) | ((stop & 0xFF) == 6) | ((stop & 0x100) != 0)
    return np.where(bad, np.float32(np.inf), rho)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--population", type=int, default=1000)
    ap.add_argument("--quantile", type=float, default=0.5)
    ap.add_argument("--max-generations", type=int, default=30)
    ap.add_argument("--max-simulations", type=int, default=20_000_000)
    ap.add_argument("--rejection-max", type=int, default=1_000_000)
    ap.add_argument("--rejection-chunk", type=int, default=250_000)
    ap.add_argument("--pairs-n", type=int, default=100_000)
    ap.add_argument("--scales", default="1,0.5,0.25,0.125", help="factors on C4's thresholds, one comparison each")
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    import _pkg
    m = _pkg.load()
    report = {"card": card(), "shape": "C4: 1e5-cell birth-death runs, b1~U(1,2), d0,d1~U(0,0.5), target = run at "
              "(1.4,0.2,0.2)", "population": a.population, "quantile": a.quantile, "runs": []}
    ctx = m.Context(0)
    opts = m.SimulationOptions(b0=1.0, b1=1.4, d0=0.2, d1=0.2, cells=100_000, save_snapshots=False)
    target = ctx.run(opts, n_runs=1, idx_begin=260, want=("hist",), hist_stride=512).hist[0].astype(np.uint64)

    mc = m.MultiContext([0])
    for scale in [float(x) for x in a.scales.split(",")]:
        thr = tuple(float(np.float32(t * scale)) for t in THR)
        entry = {"threshold_scale": scale, "thresholds": thr}
        report["runs"].append(entry)
        # ---- rejection ABC at the thresholds, chunk by chunk until M accepted draws ----
        M = a.population
        n_acc, drawn, kernel_ms, total_ms, nth = 0, 0, 0.0, 0.0, None
        idx0 = opts.idx_begin
        while drawn < a.rejection_max and nth is None:
            n = min(a.rejection_chunk, a.rejection_max - drawn)
            rates = ctx.abc_draw_priors(opts.seed, idx0 + drawn, n, **BOX)
            res = ctx.run(opts, n_runs=n, idx_begin=idx0 + drawn, want=("stop_reason", "abc_distance", "abc_accept"),
                          rates_per_run=rates, abc_target=target, abc_thresholds=thr, snapshots=False)
            ok = np.nonzero((res.abc_accept != 0) & np.isfinite(valid_rho(res.abc_distance, res.stop_reason, thr)))[0]
            if n_acc + len(ok) >= M:
                nth = drawn + int(ok[M - n_acc - 1]) + 1
            n_acc += len(ok)
            drawn += n
            kernel_ms += res.timing.kernel_ms
            total_ms += res.timing.total_ms
        entry["rejection"] = {"draws_simulated": drawn, "accepted": n_acc, "acceptance_rate": n_acc / drawn,
                               "draws_to_population": nth, "kernel_ms": kernel_ms, "call_ms_with_copies": total_ms,
                               "note": "device time covers every simulated chunk (CUDA events)"}
        print(json.dumps(entry["rejection"]), flush=True)

        # ---- ABC-SMC to the same thresholds ----
        t0 = time.perf_counter()
        r = mc.abc_smc(opts, target, thr, M, quantile=a.quantile, max_generations=a.max_generations,
                       max_simulations=a.max_simulations, **BOX)
        wall = time.perf_counter() - t0
        g = r["generations"]
        entry["smc"] = {"status": r["status"], "generations": g, "epsilon": [float(x) for x in r["epsilon"]],
                         "consumed": [int(x) for x in r["consumed"]], "simulated": [int(x) for x in r["simulated"]],
                         "ess": [float(x) for x in r["ess"]],
                         "ms_simulation": [float(x) for x in r["time_ms"][:, 0]],
                         "ms_proposal": [float(x) for x in r["time_ms"][:, 1]],
                         "ms_weights": [float(x) for x in r["time_ms"][:, 2]],
                         "total_simulated": int(r["simulated"].sum()), "total_consumed": int(r["consumed"].sum()),
                         "wall_s": wall}
        if g:
            w, th = r["weight"][-1], r["rates"][-1][:, 1:].astype(np.float64)
            entry["smc"]["posterior_mean_b1_d0_d1"] = [float(np.sum(w * th[:, k])) for k in range(3)]
        print(json.dumps(entry["smc"]), flush=True)
    mc.close()

    # ---- the weight kernel alone ----
    rng = np.random.default_rng(1)
    N = a.pairs_n

    def particles():
        return np.column_stack([np.ones(N), rng.uniform(1, 2, N), rng.uniform(0, 0.5, (N, 2))]).astype(np.float32)
    new, prev = particles(), particles()
    w = np.full(N, 1.0 / N)
    sigma = tuple(float(np.sqrt(2 * prev[:, k].var())) for k in (1, 2, 3))
    ctx.abc_smc_weights(new, prev, w, sigma, **BOX)  # warm-up: module load, buffers
    times = []
    for _ in range(5):
        t0 = time.perf_counter()
        ctx.abc_smc_weights(new, prev, w, sigma, **BOX)
        times.append((time.perf_counter() - t0) * 1e3)
    kernel = None
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                ctx.abc_smc_weights(new, prev, w, sigma, **BOX)
            torch.cuda.synchronize()
        ks = [e.device_time for e in prof.events() if "smc_pair_kernel" in e.name]
        kernel = float(np.median(ks)) / 1e3 if ks else None  # ms
    except Exception as e:  # the call times above stand on their own
        print(f"profiler: {e}", file=sys.stderr)
    pairs = float(N) * N
    report["weights_kernel"] = {"N": N, "M": N, "call_ms_median": float(np.median(times)), "call_ms_all": times,
                                "pair_kernel_ms": kernel,
                                "pairs_per_s_call": pairs / (np.median(times) / 1e3),
                                "pairs_per_s_kernel": pairs / (kernel / 1e3) if kernel else None}
    print(json.dumps(report["weights_kernel"]), flush=True)
    ctx.close()
    with open(os.path.join(a.out, "abc_smc_compare.json"), "w") as f:
        json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
