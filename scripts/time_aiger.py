"""Time AIGER conversion on the host (deepgate/aiger.py) and the GPU labelling of converted netlists.

    python scripts/time_aiger.py [--reps 5] [--out DIR]

Prints the host CPU and the card's name and power limit, then one JSON line per measurement:
  * ``convert``: read_aiger on a generated binary AIG of 1 000 000 ANDs (64 inputs, 64 latches) and on the 200 k-AND
    sequential netlist of tests/test_aiger.py (64 inputs, 512 latches, > 1 000 levels); host clock, median of --reps;
  * ``label``: label_circuits (pair draw, batching, simulation, copy back) on that 200 k-AND netlist at 32 768 random
    patterns, and on a batch of 64 converted circuits (32 ripple-carry adders and 32 array multipliers of 4 to 8 bits)
    at 32 768 random patterns and exhaustively; host clock around the call, which ends in a copy to the host, so it
    includes the GPU's work; plus simulate_counts alone on the same batch with CUDA events.  Two warm-up calls, median of
    --reps.
"""
import argparse
import json
import os
import platform
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "multi-gate-vae_b200"), ROOT, os.path.join(ROOT, "scripts"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from test_aiger import adder, multiplier, random_aig  # noqa: E402


def host_cpu():
    try:
        with open("/proc/cpuinfo") as f:
            model = next(l.split(":", 1)[1].strip() for l in f if l.startswith("model name"))
    except (OSError, StopIteration):
        model = platform.processor() or "unknown"
    return "%s (%d logical cores; the reader runs on one)" % (model, os.cpu_count())


def median_time(fn, reps, warm=1, sync=False):
    for _ in range(warm):
        fn()
    ms = []
    for _ in range(reps):
        if sync:
            torch.cuda.synchronize()
        t = time.perf_counter()
        fn()
        if sync:
            torch.cuda.synchronize()
        ms.append((time.perf_counter() - t) * 1e3)
    return float(np.median(ms)), [round(v, 3) for v in ms]


def event_time(fn, reps):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        e.record()
        e.synchronize()
        ms.append(a.elapsed_time(e))
    return float(np.median(ms)), [round(v, 3) for v in ms]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import deepgate
    from deepgate.aiger import read_aiger
    from deepgate.simulate import simulate_counts
    from deepgate.utils.dag_utils import top_sort_host
    cpu = host_cpu()
    print("host: %s" % cpu)
    lines = []

    def emit(rec):
        print(json.dumps(rec))
        lines.append(rec)

    tmp = tempfile.mkdtemp(prefix="time_aiger_")
    files = {}
    for name, (I, L, A, window, seed) in {"and1m": (64, 64, 1_000_000, 2000, 1), "seq200k": (64, 512, 200_000, 800, 3)}.items():
        data, _ = random_aig(I, L, A, window, seed)
        files[name] = os.path.join(tmp, name + ".aig")
        with open(files[name], "wb") as f:
            f.write(data)
        ms, all_ms = median_time(lambda: read_aiger(files[name], "mig"), args.reps)
        c = read_aiger(files[name], "mig")
        emit({"what": "convert", "file": name, "ands": A, "bytes": len(data), "nodes": len(c["x"]),
              "edges": len(c["edge_index"]), "host_ms": round(ms, 1), "host_ms_all": all_ms, "host": cpu})
    if not torch.cuda.is_available():
        raise SystemExit("time_aiger: no CUDA device, GPU labelling not measured")
    from time_logic_sim import card
    name, power, clock = card()
    print("card: %s, power limit %s, max SM clock %s" % (name, power, clock))
    seq = [read_aiger(files["seq200k"], "mig")]
    arith = []
    for i in range(32):
        n = 4 + i % 5
        for kind_name, text in (("adder%d_%d" % (n, i), adder(n)), ("mult%d_%d" % (n, i), multiplier(n))):
            p = os.path.join(tmp, kind_name + ".aag")
            with open(p, "w") as f:
                f.write(text)
            arith.append(read_aiger(p, "mig"))
    for label, circuits, modes in (("seq200k", seq, (False,)), ("arith64", arith, (False, True))):
        G = deepgate.circuits_to_batch([dict(c, prob=np.zeros(len(c["x"]), np.float32),
                                             tt_pair_index=np.zeros((0, 2), np.int64), tt_sim=np.zeros(0, np.float32))
                                        for c in circuits], "cuda:0")
        n = G.x.size(0)
        levels = max(int(top_sort_host(c["edge_index"].T, len(c["x"])).max()) + 1 for c in circuits)
        for exhaustive in modes:
            kw = dict(patterns=32768, exhaustive=exhaustive)
            lab_ms, lab_all = median_time(lambda: deepgate.label_circuits(circuits, "mig", "cuda:0", **kw), args.reps,
                                          warm=2, sync=True)
            sim_ms, sim_all = event_time(lambda: simulate_counts(G, "mig", **kw), args.reps)
            patterns = simulate_counts(G, "mig", **kw)[2]
            emit({"what": "label", "workload": label, "circuits": len(circuits), "N": n, "levels_max": levels,
                  "exhaustive": exhaustive, "patterns": patterns, "label_circuits_ms": round(lab_ms, 3),
                  "label_circuits_ms_all": lab_all, "simulate_counts_ms": round(sim_ms, 3),
                  "simulate_counts_ms_all": sim_all, "card": name, "power_limit": power, "max_sm_clock": clock})
        del G
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "time_aiger.jsonl"), "a") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
