"""Numpy reference of sequential simulation (deepgate.simulate_counts with ``cycles``, csrc/logic_sim.cu's seq_sim_kernel),
the oracle of tests/test_seq_sim.py.

Semantics: ``patterns`` traces, 64 per word, each starting in the reset state (reset 0: the word 0, reset 1: ~0,
uninitialised: the random-mode word of its INPUT at trace word w).  In cycle t = 0 .. C-1 every primary INPUT takes the
random-mode word of global index t * T + w (T = patterns / 64), every node is evaluated from the primary inputs and the
state, and then every latch takes the value of its next-state literal (2 u + complemented, -2 / -1 the constants).
Cycles t in [warmup, C) are counted.  Built on oracle/logic_sim.py's definitions (gate tables, levels, INPUT ranks and
INPUT words, through sim_classes_oracle._prepare); oracle/ stays as it is, so the level walk that takes given INPUT words
is here.  Plain: one level at a time, one gate function at a time.
"""
import numpy as np

import sim_classes_oracle as SO
from oracle import logic_sim as OL


def walk(net, input_rows):
    """uint64 [N, W]: every node's words, the INPUT nodes' taken from ``input_rows`` [N, W] (other rows not read)."""
    n, fn, lvl = net["n"], net["fn"], net["lvl"]
    preds_src, in_deg, in_ptr = net["preds_src"], net["in_deg"], net["in_ptr"]
    sim = np.zeros_like(input_rows)
    for l in range(int(lvl.max()) + 1 if n else 0):
        at = lvl == l
        for f in np.unique(fn[at]):
            nodes = np.flatnonzero(at & (fn == f))
            if f == "INPUT":
                sim[nodes] = input_rows[nodes]
                continue
            for d in np.unique(in_deg[nodes]):
                grp = nodes[in_deg[nodes] == d]
                ins = [sim[preds_src[in_ptr[grp] + j]] for j in range(d)]
                if f == "NOT":
                    out = ~ins[0]
                elif f == "MAJ":
                    a, b, c = ins
                    out = (a & b) | (a & c) | (b & c)
                else:
                    op = {"AND": np.bitwise_and, "OR": np.bitwise_or, "XOR": np.bitwise_xor}[f]
                    out = ins[0]
                    for x in ins[1:]:
                        out = op(out, x)
                sim[grp] = out
    return sim


def literal_words(sim, lit):
    """uint64 [len(lit), W]: the words of literals over the nodes (-2 / -1 the constants)."""
    lit = np.asarray(lit, np.int64)
    w = sim[np.maximum(lit, 0) >> 1]
    w = np.where((lit & 1)[:, None] == 1, ~w, w)
    return np.where((lit < 0)[:, None], np.where((lit == -1)[:, None], OL.M64, np.uint64(0)), w)


def simulate(code, edge_index, kind, latches=None, batch=None, pairs=None, patterns=32768, seed=0, cycles=1, warmup=0,
             words_per_pass=None):
    """Returns (ones int64 [N], diff int64 [P], samples = patterns * (cycles - warmup)).  ``latches`` int64 [L, 3]
    (INPUT node, next-state literal, reset 0 / 1 / 2 = uninitialised); ``words_per_pass`` splits the traces."""
    net, patterns = SO._prepare(code, edge_index, kind, batch, patterns, False)
    n, rank = net["n"], net["rank"]
    lat = np.zeros((0, 3), np.int64) if latches is None else np.asarray(latches, np.int64).reshape(-1, 3)
    pairs = np.zeros((2, 0), np.int64) if pairs is None else np.asarray(pairs, np.int64).reshape(2, -1)
    inputs = np.flatnonzero(net["fn"] == "INPUT")
    primary = np.setdiff1d(inputs, lat[:, 0])
    T = patterns // 64
    step = T if words_per_pass is None else int(words_per_pass)
    ones = np.zeros(n, np.int64)
    diff = np.zeros(pairs.shape[1], np.int64)
    for first in range(0, T, step):
        words = np.arange(first, min(first + step, T))
        state = np.zeros((len(lat), words.size), np.uint64)
        state[lat[:, 2] == 1] = OL.M64
        un = lat[:, 2] == 2
        state[un] = OL.input_words(rank[lat[un, 0]], words, seed, False)
        for t in range(cycles):
            rows = np.zeros((n, words.size), np.uint64)
            rows[primary] = OL.input_words(rank[primary], t * T + words, seed, False)
            rows[lat[:, 0]] = state
            sim = walk(net, rows)
            if t >= warmup:
                ones += OL.popcount(sim)
                if pairs.shape[1]:
                    diff += OL.popcount(sim[pairs[0]] ^ sim[pairs[1]])
            state = literal_words(sim, lat[:, 1])
    return ones, diff, patterns * (cycles - warmup)
