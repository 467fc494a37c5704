"""Time sequential simulation (simulate_counts with ``cycles``, csrc/logic_sim.cu's seq_sim_kernel) on the GPU.

    python scripts/time_seq_sim.py [--reps 5] [--out DIR]

Workloads, AIGs generated as tests/test_aiger.py does (resets 0):
  * seq200k: the 200 k-AND netlist with 64 inputs and 512 latches (> 1 000 levels);
  * and1m: the 1 000 000-AND file of scripts/time_aiger.py (64 inputs, 64 latches);
  * small64: a batch of 64 sequential AIGs of cfg2 size (16 to 64 inputs, 8 to 32 latches, 500 to 1 500 ANDs).
Each at 32 768 traces and C = 16 and 64 cycles (warm-up 0), at simulate_counts' default 4 GiB buffer bound.  CUDA events
around the whole simulate_counts call, median of --reps after two warm-up calls; the combinational simulate_counts at
32 768 patterns on the same batch is the one-cycle reference point.  Algorithmic bytes = cycles x traces / 8 x (N + E):
every node's words written and every edge's source words read once per cycle, over HBM's 7.7 TB/s (a bound, not what the
kernel moves: small batches stay in L2).  Prints the card's name, power limit and max SM clock, then one JSON line per
measurement and a table.
"""
import argparse
import json
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "multi-gate-vae_b200"), ROOT, os.path.join(ROOT, "scripts"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from test_aiger import random_aig  # noqa: E402
from time_aiger import event_time  # noqa: E402

TRACES, CYCLES = 32768, (16, 64)


def workloads(tmp):
    from deepgate.aiger import read_aiger
    out = {}
    specs = {"seq200k": [(64, 512, 200_000, 800, 3)], "and1m": [(64, 64, 1_000_000, 2000, 1)],
             "small64": [(16 + i % 49, 8 + i % 25, 500 + (i * 97) % 1001, 50, 100 + i) for i in range(64)]}
    for name, spec in specs.items():
        circuits = []
        for j, (I, L, A, window, seed) in enumerate(spec):
            path = os.path.join(tmp, "%s_%d.aig" % (name, j))
            with open(path, "wb") as f:
                f.write(random_aig(I, L, A, window, seed)[0])
            circuits.append(read_aiger(path, "aig"))
        out[name] = circuits
    return out


def measure(reps, tmp):
    import deepgate
    from deepgate.simulate import _Sim, _batch_latches, simulate_counts
    from time_logic_sim import card
    name, power, clock = card()
    recs = []
    for label, circuits in workloads(tmp).items():
        G = deepgate.circuits_to_batch([dict(c, prob=np.zeros(len(c["x"]), np.float32), tt_sim=np.zeros(0, np.float32),
                                             tt_pair_index=np.zeros((0, 2), np.int64)) for c in circuits], "cuda:0")
        lat = _batch_latches(circuits)
        n, e = G.x.size(0), G.edge_index.size(1)
        base = {"workload": label, "circuits": len(circuits), "N": n, "E": e, "latches": len(lat), "traces": TRACES,
                "card": name, "power_limit": power, "max_sm_clock": clock}
        s = _Sim(G, "aig", TRACES, 0, False, 2 ** 32)
        ms, all_ms = event_time(lambda: simulate_counts(G, "aig", patterns=TRACES), reps)
        recs.append(dict(base, what="combinational", passes=-(-s.total // s.words_per_pass()), ms=round(ms, 3),
                         ms_all=all_ms))
        for C in CYCLES:
            kw = dict(patterns=TRACES, cycles=C, latches=lat)
            s = _Sim(G, "aig", TRACES, 0, False, 2 ** 32, C, 0, lat)
            passes = -(-s.total // s.words_per_pass())
            ms, all_ms = event_time(lambda: simulate_counts(G, "aig", **kw), reps)
            byts = C * TRACES / 8 * (n + e)
            recs.append(dict(base, what="sequential", cycles=C, passes=passes, ms=round(ms, 3), ms_all=all_ms,
                             ms_per_cycle=round(ms / C, 4), algorithmic_GB=round(byts / 1e9, 2),
                             TBps=round(byts / ms / 1e9, 3), share_of_7_7TBps=round(byts / ms / 1e9 / 7.7, 3)))
        del G
        torch.cuda.empty_cache()
    return recs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_seq_sim: no CUDA device, nothing measured")
    from time_logic_sim import card
    print("card: %s, power limit %s, max SM clock %s" % tuple(card()))
    recs = measure(args.reps, tempfile.mkdtemp(prefix="time_seq_sim_"))
    for rec in recs:
        print(json.dumps(rec))
    print("| workload | N | latches | C | passes | ms per call | ms per cycle | algorithmic TB/s |")
    print("|---|---|---|---|---|---|---|---|")
    for r in recs:
        if r["what"] == "combinational":
            print("| %s | %d | %d | combinational | %d | %.3f | | |" % (r["workload"], r["N"], r["latches"], r["passes"],
                                                                      r["ms"]))
        else:
            print("| %s | %d | %d | %d | %d | %.3f | %.3f | %.3f |" % (r["workload"], r["N"], r["latches"], r["cycles"],
                                                                     r["passes"], r["ms"], r["ms_per_cycle"], r["TBps"]))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "time_seq_sim.jsonl"), "a") as f:
            for rec in recs:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
