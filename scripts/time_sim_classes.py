"""Time functional equivalence classes (deepgate.equivalence_classes, csrc/sim_classes.cu) against the simulation alone.

    python scripts/time_sim_classes.py [--patterns 32768] [--reps 5] [--workloads cfg2,cfg5-k64] [--out DIR]

Prints the card name and power limit, then per workload (bench.py's circuit draws, as scripts/time_logic_sim.py) and
buffer bound ``max_bytes``:
  * ms of simulate_counts and of equivalence_classes on the same batch: CUDA events around the whole call, two warm-up
    calls, median of --reps; the difference is what the classes add;
  * algorithmic bytes / time of the classes call against 7.7 TB/s.  Bytes: the simulation passes as in time_logic_sim.py
    (run twice when there is more than one pass: hash, then check), 8 N W for the signature read, 16 M W for the check
    (M = nodes that are not their class representative), and 76 N for the key, head and scatter kernels; the radix sort and
    scan inside cub are not counted;
  * classes with more than one node, the nodes in them, and n_split;
and, for cfg2, how many of the pairs that label_circuits draws today (64 uniform random pairs per circuit) have a
truth-table distance of exactly 0 or 1, against the pairs drawn with class_pairs=64.  One JSON line per measurement.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "multi-gate-vae_b200"), ROOT, os.path.join(ROOT, "scripts")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from time_logic_sim import HBM_BYTES_PER_S, WORKLOADS, algorithmic_bytes, card  # noqa: E402


def timed(fn, reps):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    ms, out = [], None
    for _ in range(reps):
        a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        e.record()
        e.synchronize()
        ms.append(a.elapsed_time(e))
    return float(np.median(ms)), ms, out


def extreme_pairs(circuits, kind, class_pairs, patterns):
    """Pairs drawn as label_circuits draws them, and how many have distance exactly 0 or 1."""
    import deepgate
    cs = [dict(c) for c in circuits]
    for c in cs:
        c.pop("tt_pair_index", None)
    labelled = deepgate.label_circuits(cs, kind, "cuda:0", n_pairs=64, class_pairs=class_pairs, patterns=patterns)
    tt = np.concatenate([c["tt_sim"] for c in labelled])
    return {"class_pairs": class_pairs, "pairs": int(tt.size), "dist_0": int((tt == 0).sum()), "dist_1": int((tt == 1).sum())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--patterns", type=int, default=32768)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--workloads", default="cfg2,cfg5-k64")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_sim_classes: no CUDA device")
    import deepgate
    from deepgate import synth
    from deepgate.simulate import SLICE_WORDS, simulate_counts
    name, power, clock = card()
    print("card: %s, power limit %s, max SM clock %s" % (name, power, clock))
    bounds = {"cfg2": [2 ** 32], "cfg5-k64": [2 ** 32, 2 ** 35]}
    lines = []
    for wl in args.workloads.split(","):
        kind, mix, b, n_pi, n_gates, window, cfg = WORKLOADS[wl]
        circuits = synth.make_circuits(mix, b, n_pi, n_gates, cfg=cfg, window=window)
        G = deepgate.circuits_to_batch(circuits, "cuda:0")
        n, P = G.x.size(0), G.tt_pair_index.size(1)
        total = args.patterns // 64
        for mb in bounds[wl]:
            W = min(total, mb // (8 * n) // SLICE_WORDS * SLICE_WORDS)
            passes = -(-total // W)
            sim_ms, sim_all, _ = timed(lambda: simulate_counts(G, kind, patterns=args.patterns, max_bytes=mb), args.reps)
            cls_ms, cls_all, (rep, comp, n_split) = timed(
                lambda: deepgate.equivalence_classes(G, kind, patterns=args.patterns, max_bytes=mb), args.reps)
            rep = rep.cpu().numpy()
            size = np.bincount(rep, minlength=n)
            members = int((rep != np.arange(n)).sum())
            nbytes = (algorithmic_bytes(G, total, W, 0) * (1 if passes == 1 else 2) + 8.0 * n * total
                      + 16.0 * members * total + 76.0 * n)
            rec = {"workload": wl, "card": name, "power_limit": power, "N": n, "patterns": args.patterns, "max_bytes": mb,
                   "words_per_pass": W, "passes": passes, "simulate_counts_ms": round(sim_ms, 3),
                   "equivalence_classes_ms": round(cls_ms, 3), "added_ms": round(cls_ms - sim_ms, 3),
                   "simulate_counts_ms_all": [round(v, 3) for v in sim_all],
                   "equivalence_classes_ms_all": [round(v, 3) for v in cls_all],
                   "algorithmic_bytes": nbytes, "bytes_per_s": nbytes / (cls_ms / 1e3),
                   "hbm_fraction": nbytes / (cls_ms / 1e3) / HBM_BYTES_PER_S,
                   "classes_gt1": int((size > 1).sum()), "nodes_in_classes_gt1": int(size[size > 1].sum()),
                   "complemented": int(comp.sum()), "n_split": n_split}
            print(json.dumps(rec))
            lines.append(rec)
        if wl == "cfg2":
            for k in (0, 64):
                rec = dict(workload=wl, card=name, power_limit=power, **extreme_pairs(circuits, kind, k, args.patterns))
                print(json.dumps(rec))
                lines.append(rec)
        del G
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "time_sim_classes.jsonl"), "a") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
