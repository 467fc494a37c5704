"""Time circuit labelling by logic simulation (deepgate.simulate, csrc/logic_sim.cu) on one GPU.

    python scripts/time_logic_sim.py [--patterns 32768] [--reps 5] [--workloads cfg2,cfg5-k64] [--out DIR]

Prints the card name and power limit, then per workload (bench.py's circuit draws: cfg2 = 64 AIG circuits of 500-1500
gates; cfg5-k64 = 64 MIG circuits of 100 k gates, 687 levels) and buffer bound ``max_bytes``:
  * ms per batch: CUDA events around simulate_counts (validation + every pass) after two warm-up calls, median of --reps;
  * pattern.gates/s = patterns x N / time;
  * algorithmic bytes / time against 7.7 TB/s HBM.  Bytes per pass: 8 W sum(fan-in + 1) for the simulation, 8 N ceil(W / 4) for
    the count atomics and 16 W P for the pair pass (W = words of the pass, P = pairs);
and, for cfg2, the numpy oracle's time on the host cores.  One JSON line per measurement; --out also writes them there.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "multi-gate-vae_b200"), ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

HBM_BYTES_PER_S = 7.7e12
WORKLOADS = {    # bench.py WORKLOADS: kind, mix, circuits, n_pi, n_gates, window, cfg
    "cfg2": ("aig", "aig", 64, (16, 64), (500, 1500), None, 2),
    "cfg5-k64": ("mig", "mig", 64, 16, 100000, 880, 5),
}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        return [s.strip() for s in q.split(",")]
    except Exception as e:                                  # noqa: BLE001
        return [torch.cuda.get_device_name(0), "power limit unknown (%s)" % e, ""]


def algorithmic_bytes(G, total_words, W, P):
    n = G.x.size(0)
    fanin_plus_one = float(n + G.edge_index.size(1))
    out = 0.0
    for first in range(0, total_words, W):
        w = min(W, total_words - first)
        out += 8.0 * w * fanin_plus_one + 8.0 * n * ((w + 3) // 4) + 16.0 * w * P
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--patterns", type=int, default=32768)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--workloads", default="cfg2,cfg5-k64")
    ap.add_argument("--max-bytes", default="4294967296,34359738368", help="comma-separated buffer bounds to time")
    ap.add_argument("--oracle", type=int, default=1, help="also time the numpy oracle on cfg2")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_logic_sim: no CUDA device")
    import deepgate
    from deepgate import synth
    from deepgate.simulate import simulate_counts, SLICE_WORDS
    from oracle import logic_sim as OL
    name, power, clock = card()
    lib = os.environ.get("MGV_B200_LIB", "default build")
    print("card: %s, power limit %s, max SM clock %s, library %s" % (name, power, clock, lib))
    lines = []
    for wl in args.workloads.split(","):
        kind, mix, b, n_pi, n_gates, window, cfg = WORKLOADS[wl]
        t0 = time.time()
        circuits = synth.make_circuits(mix, b, n_pi, n_gates, cfg=cfg, window=window)
        G = deepgate.circuits_to_batch(circuits, "cuda:0")
        n, P = G.x.size(0), G.tt_pair_index.size(1)
        L = int(G.forward_level.max()) + 1
        print("%s: N = %d, E = %d, L = %d, P = %d (built in %.1f s)" % (wl, n, G.edge_index.size(1), L, P, time.time() - t0))
        total = args.patterns // 64
        for mb in (int(v) for v in args.max_bytes.split(",")):
            W = min(total, mb // (8 * n) // SLICE_WORDS * SLICE_WORDS)
            for _ in range(2):
                simulate_counts(G, kind, patterns=args.patterns, max_bytes=mb)
            torch.cuda.synchronize()
            ms = []
            for _ in range(args.reps):
                a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                ones, diff, _ = simulate_counts(G, kind, patterns=args.patterns, max_bytes=mb)
                e.record()
                e.synchronize()
                ms.append(a.elapsed_time(e))
            t = float(np.median(ms)) / 1e3
            nbytes = algorithmic_bytes(G, total, W, P)
            rec = {"workload": wl, "card": name, "power_limit": power, "library": lib, "N": n, "L": L, "P": P,
                   "patterns": args.patterns, "max_bytes": mb, "words_per_pass": W, "passes": -(-total // W),
                   "ctas_per_pass": -(-W // SLICE_WORDS), "ms": round(t * 1e3, 3), "ms_all": [round(v, 3) for v in ms],
                   "pattern_gates_per_s": args.patterns * n / t, "algorithmic_bytes": nbytes,
                   "bytes_per_s": nbytes / t, "hbm_fraction": nbytes / t / HBM_BYTES_PER_S,
                   "mean_prob": float(ones.double().mean() / args.patterns)}
            print(json.dumps(rec))
            lines.append(rec)
        if wl == "cfg2" and args.oracle:
            host = G.to("cpu")
            t0 = time.time()
            OL.simulate(host.gate.reshape(-1).long().numpy(), host.edge_index.numpy(), kind, batch=host.batch.numpy(),
                        pairs=host.tt_pair_index.numpy(), patterns=args.patterns)
            rec = {"workload": wl, "oracle_s": round(time.time() - t0, 3), "host_cores": os.cpu_count(),
                   "note": "numpy, one process"}
            print(json.dumps(rec))
            lines.append(rec)
        del G
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "time_logic_sim.jsonl"), "a") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
