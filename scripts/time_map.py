"""Time the AIG -> MIG / XMG / XAG mapping (deepgate/mapping.py, csrc/map_cuts.cu).

    python scripts/time_map.py [--reps 5] [--out DIR]

Prints the card's name and power limit, then one JSON line per (workload, kind):
  * workloads: the 1 000 000-AND binary AIG of tests/test_aiger.py::test_million_and_binary_converts, the 200 k-AND
    sequential netlist (> 1 000 levels), and the cfg2 AIG batch (64 synthetic circuits of 500 to 1 500 gates);
  * ``gpu_ms``: enumeration and cover (mgv_map_cuts + mgv_map_cover) under CUDA events;
  * ``emit_ms``: the host emission of the mapped dicts from the per-node arrays; ``map_circuits_ms``: the whole call
    (batching and level schedule, kernels, copy back, emission), host clock;
  * ``oracle_ms``: tests/map_oracle.py on one cfg2 circuit, host clock;
  * ANDs in, nodes and gates of each type out.
One warm-up, median of --reps.
"""
import argparse
import json
import os
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "multi-gate-vae_b200"), ROOT, os.path.join(ROOT, "scripts"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from test_aiger import random_aig  # noqa: E402
from time_aiger import event_time, median_time  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_map: no CUDA device, nothing measured")
    from deepgate import mapping as MP, synth
    from deepgate.aiger import read_aiger
    import map_oracle as MO
    from time_logic_sim import card
    name, power, clock = card()
    print("card: %s, power limit %s, max SM clock %s" % (name, power, clock))
    tmp = tempfile.mkdtemp(prefix="time_map_")
    workloads = {}
    for label, (I, L, A, window, seed) in {"and1m": (64, 64, 1_000_000, 2000, 1), "seq200k": (64, 512, 200_000, 800, 3)}.items():
        path = os.path.join(tmp, label + ".aig")
        with open(path, "wb") as f:
            f.write(random_aig(I, L, A, window, seed)[0])
        workloads[label] = [read_aiger(path, "aig")]
    workloads["cfg2"] = synth.make_circuits("aig", 64, (16, 64), (500, 1500), cfg=2)
    small = workloads["cfg2"][0]
    lines = []
    for label, circuits in workloads.items():
        ands = sum(int((c["x"][:, 1] == 1).sum()) for c in circuits)
        for kind in ("mig", "xmg", "xag"):
            b = MP._Batch(circuits, kind, "cuda:0")
            gpu_ms, gpu_all = event_time(b.run, args.reps)
            arrays = b.arrays()
            levels = len(b.levels)
            del b
            emit_ms, emit_all = median_time(lambda: [MP.emit(c, kind, a) for c, a in zip(circuits, arrays)], args.reps)
            map_ms, map_all = median_time(lambda: MP.map_circuits(circuits, kind, "cuda:0"), args.reps, sync=True)
            oracle_ms, _ = median_time(lambda: MO.map_circuit(small, kind), 1, warm=0)
            mapped = MP.map_circuits(circuits, kind, "cuda:0")
            rec = {"workload": label, "kind": kind, "circuits": len(circuits), "ands_in": ands, "and_levels": levels,
                   "nodes_out": sum(len(m["x"]) for m in mapped), "gates_out": MP.gate_counts(mapped, kind),
                   "gpu_ms": round(gpu_ms, 3), "gpu_ms_all": gpu_all, "emit_ms": round(emit_ms, 2),
                   "map_circuits_ms": round(map_ms, 1), "map_circuits_ms_all": map_all,
                   "oracle_ms_one_cfg2_circuit": round(oracle_ms, 1), "oracle_circuit_ands": int((small["x"][:, 1] == 1).sum()),
                   "card": name, "power_limit": power, "max_sm_clock": clock}
            print(json.dumps(rec), flush=True)
            lines.append(rec)
            torch.cuda.empty_cache()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "time_map.jsonl"), "a") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
