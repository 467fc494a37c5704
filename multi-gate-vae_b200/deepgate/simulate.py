"""Circuit labels by bit-parallel logic simulation on the GPU (csrc/logic_sim.cu): ``prob`` (probability that a node is 1
under random inputs) and the truth-table distance of node pairs (``tt_sim`` in a batch, ``tt_dis`` in ``labels.npz``).

    prob, tt_dis = simulate(G, "mig")                       # a CUDA batch, e.g. circuits_to_batch(circuits, "cuda")
    labelled = label_circuits(circuits, "mig", "cuda:0")    # synth-style circuit dicts -> copies with labels
    write_npz(labelled, "graphs.npz", "labels.npz", "mig")  # the reference's on-disk layouts, read back by NpzParser
    python -m deepgate.simulate --graphs graphs.npz --type mig --out DIR

Gate functions by code: AIG {0 INPUT, 1 AND, 2 NOT}; MIG / XMG / XAG {0 INPUT, 1 MAJ, 2 NOT, 3 AND, 4 OR, 5 XOR}.  AND, OR
and XOR reduce over all their predecessors, NOT takes one, MAJ three.  Random mode: ``patterns`` (a multiple of 64) patterns;
word w of an INPUT is a splitmix64 hash of (seed, the INPUT's rank among the INPUTs of its own circuit, w), so a circuit's
labels do not depend on the batch it sits in or on how the words are split into passes.  Exhaustive mode: every input
assignment of the largest circuit (K inputs, K <= 24), ``max(64, 2^K)`` patterns: exact probabilities.  The counts are
integers, so results are deterministic.  There is no CPU path; ``oracle/logic_sim.py`` is the numpy reference of the tests.

The package exports ``simulate``, ``simulate_counts``, ``label_circuits`` and ``write_npz`` as ``deepgate.<name>``; the package
attribute ``deepgate.simulate`` is therefore the function, and the module is reached as ``from deepgate.simulate import ...``
or ``sys.modules["deepgate.simulate"]``.
"""
import argparse
import ctypes
import os

import numpy as np
import torch

from . import _native as nat
from .schedule import schedule_for_batch

_F = {"NONE": 0, "INPUT": 1, "AND": 2, "OR": 3, "XOR": 4, "NOT": 5, "MAJ": 6}       # MGV_FN_* (include/mgv_b200.h)
_AIG = ("INPUT", "AND", "NOT")                                                    # dg_ae_model_aig.py codes
_GATE_TO_INDEX = ("INPUT", "MAJ", "NOT", "AND", "OR", "XOR")                      # reference parser.py:133
CODE_TABLES = {"aig": _AIG, "mig": _GATE_TO_INDEX, "xmg": _GATE_TO_INDEX, "xag": _GATE_TO_INDEX}
MAX_EXHAUSTIVE_INPUTS = 24
SLICE_WORDS = 4                          # words per CTA slice of the kernel: a pass's word count is rounded down to it


def _fn_table(kind):
    if kind not in CODE_TABLES:
        raise ValueError("kind must be one of %s, got %r" % (sorted(CODE_TABLES), kind))
    names = CODE_TABLES[kind]
    return (ctypes.c_int32 * nat.NCODE)(*[_F[names[c]] if c < len(names) else _F["NONE"] for c in range(nat.NCODE)])


def _input_ranks(G, code):
    """Rank of every INPUT among the INPUTs of its circuit (``G.batch`` / ``G.ptr``; neither = one circuit), and the
    largest INPUT count of any circuit.  Runs where the batch lives."""
    n = code.numel()
    batch = getattr(G, "batch", None)
    if batch is None or batch.numel() != n:
        ptr = getattr(G, "ptr", None)
        if ptr is not None and int(ptr[-1]) == n:
            batch = torch.repeat_interleave(torch.arange(ptr.numel() - 1, device=code.device), (ptr[1:] - ptr[:-1]).to(code.device))
        else:
            batch = torch.zeros(n, dtype=torch.long, device=code.device)
    batch = batch.to(code.device, torch.long)
    is_in = (code == 0).to(torch.long)
    per = torch.zeros(int(batch.max()) + 1 if n else 1, dtype=torch.long, device=code.device).index_add_(0, batch, is_in)
    base = torch.cumsum(per, 0) - per
    rank = torch.cumsum(is_in, 0) - 1 - base[batch]
    return rank.to(torch.int32).contiguous(), int(per.max()) if n else 0


def simulate_counts(G, kind, patterns=32768, seed=0, exhaustive=False, max_bytes=2 ** 32):
    """Integer counts behind ``simulate``: (ones int64 [N], diff int64 [P], patterns) on the batch's device, ``ones[v]`` =
    patterns where node v is 1, ``diff[p]`` = patterns where the two nodes of ``G.tt_pair_index[:, p]`` differ."""
    table = _fn_table(kind)
    if not exhaustive and (int(patterns) <= 0 or int(patterns) % 64):
        raise ValueError("patterns must be a positive multiple of 64, got %r" % (patterns,))
    rank, k = _input_ranks(G, G.gate.reshape(-1).to(torch.int32))
    if exhaustive and k > MAX_EXHAUSTIVE_INPUTS:
        raise ValueError("exhaustive simulation of a circuit with %d inputs (at most %d)" % (k, MAX_EXHAUSTIVE_INPUTS))
    if not G.edge_index.is_cuda:
        raise RuntimeError("mgv_b200: the batch must be on a CUDA device (no CPU path); call batch.to('cuda')")
    sch = schedule_for_batch(G)
    dev, n = sch.device, sch.N
    patterns = max(64, 1 << k) if exhaustive else int(patterns)
    total = patterns // 64
    pairs = getattr(G, "tt_pair_index", None)
    pairs = (pairs if pairs is not None else torch.zeros(2, 0, dtype=torch.long, device=dev)).to(dev, torch.int64).contiguous()
    P = pairs.size(1)
    ones = torch.zeros(n, dtype=torch.int64, device=dev)
    diff = torch.zeros(P, dtype=torch.int64, device=dev)
    if n == 0:
        return ones, diff, patterns
    wmax = int(max_bytes) // (8 * n) // SLICE_WORDS * SLICE_WORDS
    if wmax < 1:
        raise ValueError("max_bytes = %d is below one 32-byte slice per node (%d nodes)" % (max_bytes, n))
    W = min(total, wmax)
    lib = nat.lib()
    st = nat.stream_of(dev)
    with nat.on_device(dev):
        level = sch.level.reshape(-1).to(torch.int32).contiguous()
        ws = nat.workspace(16, dev)
        nat.check(lib.mgv_logic_sim_validate(sch.c_struct(), nat.ptr(sch.code), nat.ptr(level), table, nat.ptr(pairs), P,
                                             nat.ptr(ws), ws.numel(), st), "mgv_logic_sim_validate")
        sim = nat.workspace(lib.mgv_logic_sim_bytes(n, W), dev)
        for first in range(0, total, W):
            w = min(W, total - first)
            nat.check(lib.mgv_logic_sim_pass(sch.c_struct(), nat.ptr(sch.code), nat.ptr(rank), table,
                                             1 if exhaustive else 0, int(seed) & (2 ** 64 - 1), first, w, nat.ptr(sim),
                                             nat.ptr(ones), nat.ptr(pairs), P, nat.ptr(diff), st), "mgv_logic_sim_pass")
    return ones, diff, patterns


def simulate(G, kind, patterns=32768, seed=0, exhaustive=False, max_bytes=2 ** 32):
    """Signal probability and pair truth-table distance of a CUDA batch ``G``: (prob float32 [N, 1], tt_dis float32 [P]).
    ``kind`` picks the code table ("aig", "mig", "xmg", "xag"); ``max_bytes`` bounds the simulation buffer (N x words x
    8 bytes per pass; more passes when it is smaller).  A pass runs one CTA per 4 words, so a bound that leaves fewer than
    ~600 words per pass (148 SMs) idles most of the GPU: raise it for batches of millions of nodes (DESIGN.md §4.7).  Raises ``RuntimeError`` naming the first malformed node or pair."""
    ones, diff, patterns = simulate_counts(G, kind, patterns, seed, exhaustive, max_bytes)
    prob = (ones.double() / patterns).float().reshape(-1, 1)
    return prob, (diff.double() / patterns).float()


def _pairs_for(c, index, n_pairs, seed):
    tpi = c.get("tt_pair_index")
    if tpi is not None and len(tpi) > 0:
        return np.asarray(tpi, dtype=np.int64).reshape(-1, 2)
    n = len(c["x"])
    if n < 2:
        return np.zeros((0, 2), dtype=np.int64)
    rng = np.random.default_rng([int(seed) & (2 ** 63 - 1), index])
    a = rng.integers(0, n, size=n_pairs)
    b = rng.integers(0, n - 1, size=n_pairs)
    b = b + (b >= a)                                    # distinct from a
    return np.stack([a, b], axis=1).astype(np.int64)


def label_circuits(circuits, kind, device, batch_size=64, n_pairs=64, **simulate_kw):
    """Copies of synth-style circuit dicts (``x`` with the gate code in column 1, ``edge_index`` [E, 2]) with ``prob`` [N],
    ``tt_pair_index`` [P, 2] and ``tt_sim`` [P] (the truth-table DISTANCE, what the func loss consumes) filled in.  A circuit's
    non-empty ``tt_pair_index`` is kept; otherwise ``n_pairs`` pairs of distinct nodes are drawn with a generator seeded from
    ``seed`` and the circuit's index.  Circuits are simulated ``batch_size`` at a time on ``device``."""
    from .parser_func_others import circuits_to_batch
    seed = simulate_kw.get("seed", 0)
    out = []
    for i0 in range(0, len(circuits), batch_size):
        chunk = []
        for j, c in enumerate(circuits[i0:i0 + batch_size]):
            c = dict(c)
            c["tt_pair_index"] = _pairs_for(c, i0 + j, n_pairs, seed)
            c["prob"] = np.zeros(len(c["x"]), dtype=np.float32)
            c["tt_sim"] = np.zeros(len(c["tt_pair_index"]), dtype=np.float32)
            chunk.append(c)
        G = circuits_to_batch(chunk, device)
        prob, tt = simulate(G, kind, **simulate_kw)
        prob, tt = prob.reshape(-1).cpu().numpy(), tt.cpu().numpy()
        n0 = p0 = 0
        for c in chunk:
            n, p = len(c["x"]), len(c["tt_pair_index"])
            c["prob"], c["tt_sim"] = prob[n0:n0 + n].copy(), tt[p0:p0 + p].copy()
            n0, p0 = n0 + n, p0 + p
            out.append(c)
    return out


def write_npz(circuits, graphs_path, labels_path, kind):
    """Write labelled circuits in the reference's on-disk layouts (what ``NpzParser`` reads):
      * ``aig``: everything in ``graphs.npz`` -- ``x``, ``edge_index`` [2, E], ``tt_sim``, ``tt_pair_index`` [2, P], ``prob``,
        ``gate`` [N, 1]; ``labels_path`` is not written (pass None);
      * ``mig`` / ``xmg`` / ``xag``: ``x`` and ``edge_index`` [E, 2] in ``graphs.npz``; ``tt_dis``, ``tt_pair_index`` [P, 2]
        and ``prob`` in ``labels.npz``.
    Circuits are stored under their ``name`` or ``c<index>``.  Returns (graphs_path, labels_path to give NpzParser)."""
    _fn_table(kind)
    graphs, labels = {}, {}
    for i, c in enumerate(circuits):
        name = c.get("name") or "c%05d" % i
        x = np.asarray(c["x"])
        ei = np.asarray(c["edge_index"], dtype=np.int64).reshape(-1, 2)
        tpi = np.asarray(c["tt_pair_index"], dtype=np.int64).reshape(-1, 2)
        prob = np.asarray(c["prob"], dtype=np.float32).reshape(-1)
        tt = np.asarray(c["tt_sim"], dtype=np.float32).reshape(-1)
        if kind == "aig":
            graphs[name] = {"x": x, "edge_index": ei.T.copy(), "tt_sim": tt, "tt_pair_index": tpi.T.copy(), "prob": prob,
                            "gate": x[:, 1:2].copy()}
        else:
            graphs[name] = {"x": x, "edge_index": ei}
            labels[name] = {"tt_dis": tt, "tt_pair_index": tpi, "prob": prob}
    np.savez(graphs_path, circuits=np.array(graphs, dtype=object))
    if kind == "aig":
        return graphs_path, graphs_path
    np.savez(labels_path, labels=np.array(labels, dtype=object))
    return graphs_path, labels_path


def read_circuits(graphs_path, kind):
    """Circuit dicts (``x``, ``edge_index`` [E, 2], ``name``, and ``tt_pair_index`` [P, 2] where the file has pairs) from a
    reference ``graphs.npz`` of either layout."""
    stored = np.load(graphs_path, allow_pickle=True)["circuits"].item()
    out = []
    for name, g in stored.items():
        ei = np.asarray(g["edge_index"], dtype=np.int64)
        c = {"name": name, "x": np.asarray(g["x"])}
        c["edge_index"] = ei.T.copy() if kind == "aig" else ei.reshape(-1, 2)
        if "tt_pair_index" in g:
            tpi = np.asarray(g["tt_pair_index"], dtype=np.int64)
            c["tt_pair_index"] = tpi.T.copy() if kind == "aig" else tpi.reshape(-1, 2)
        out.append(c)
    return out


def main(argv=None):
    ap = argparse.ArgumentParser(prog="python -m deepgate.simulate",
                                 description="Label the circuits of a graphs.npz by logic simulation on cuda:0 and write "
                                             "DIR/graphs.npz (+ DIR/labels.npz for mig / xmg / xag), readable by NpzParser.")
    ap.add_argument("--graphs", required=True, help="input graphs.npz (the reference layout of --type)")
    ap.add_argument("--type", required=True, choices=sorted(CODE_TABLES))
    ap.add_argument("--out", required=True, help="output directory")
    ap.add_argument("--patterns", type=int, default=32768, help="random patterns, a multiple of 64")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--exhaustive", action="store_true", help="all input assignments (circuits of at most 24 inputs)")
    ap.add_argument("--pairs", type=int, default=64, help="node pairs drawn per circuit that has none")
    args = ap.parse_args(argv)
    circuits = read_circuits(args.graphs, args.type)
    labelled = label_circuits(circuits, args.type, "cuda:0", n_pairs=args.pairs, patterns=args.patterns, seed=args.seed,
                              exhaustive=args.exhaustive)
    os.makedirs(args.out, exist_ok=True)
    gp, lp = write_npz(labelled, os.path.join(args.out, "graphs.npz"), os.path.join(args.out, "labels.npz"), args.type)
    print("labelled %d circuits -> %s%s" % (len(labelled), gp, "" if lp == gp else ", " + lp))


if __name__ == "__main__":
    main()
