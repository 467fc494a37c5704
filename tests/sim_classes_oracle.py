"""Numpy reference of deepgate.equivalence_classes (csrc/sim_classes.cu), the oracle of tests/test_sim_classes.py.

Built on oracle/logic_sim.py's definitions (gate tables, levels, INPUT ranks and INPUT words); it keeps every node's words,
which oracle/logic_sim.simulate folds into counts inside its pass loop.  Plain: one level at a time, one gate function
at a time.
"""
import numpy as np

from oracle import logic_sim as OL


def _prepare(code, edge_index, kind, batch, patterns, exhaustive):
    """Checked inputs and predecessor lists of one simulation (a dict for ``pass_words``) and the pattern count."""
    code = np.asarray(code, np.int64).reshape(-1)
    n = code.size
    ei = np.asarray(edge_index, np.int64).reshape(2, -1)
    batch = np.zeros(n, np.int64) if batch is None else np.asarray(batch, np.int64)
    table = OL.CODE_TABLES[kind]
    fn = np.array([table.get(int(c), "NONE") for c in code])
    if (fn == "NONE").any():
        raise ValueError("undefined gate code at node %d" % int(np.flatnonzero(fn == "NONE")[0]))
    if exhaustive:
        k = int(np.bincount(batch[code == 0]).max()) if (code == 0).any() else 0
        if k > 24:
            raise ValueError("exhaustive simulation of %d inputs" % k)
        patterns = max(64, 1 << k)
    if patterns <= 0 or patterns % 64:
        raise ValueError("patterns must be a positive multiple of 64")
    order = np.argsort(ei[1], kind="stable")                         # predecessors by node, ascending edge id
    in_deg = np.bincount(ei[1], minlength=n)
    in_ptr = np.zeros(n + 1, np.int64)
    np.cumsum(in_deg, out=in_ptr[1:])
    net = {"n": n, "batch": batch, "fn": fn, "rank": OL.input_ranks(code, batch), "lvl": OL.levels(ei, n),
           "preds_src": ei[0][order], "in_deg": in_deg, "in_ptr": in_ptr}
    return net, patterns


def pass_words(net, words, seed, exhaustive):
    """uint64 [N, len(words)]: every node's value on the global words ``words`` of the patterns."""
    n, fn, lvl, rank = net["n"], net["fn"], net["lvl"], net["rank"]
    preds_src, in_deg, in_ptr = net["preds_src"], net["in_deg"], net["in_ptr"]
    sim = np.zeros((n, words.size), np.uint64)
    for l in range(int(lvl.max()) + 1 if n else 0):
        at = lvl == l
        for f in np.unique(fn[at]):
            nodes = np.flatnonzero(at & (fn == f))
            if f == "INPUT":
                sim[nodes] = OL.input_words(rank[nodes], words, seed, exhaustive)
                continue
            for d in np.unique(in_deg[nodes]):
                grp = nodes[in_deg[nodes] == d]
                ins = [sim[preds_src[in_ptr[grp] + j]] for j in range(d)]
                if f == "NOT":
                    assert d == 1
                    out = ~ins[0]
                elif f == "MAJ":
                    assert d == 3
                    a, b, c = ins
                    out = (a & b) | (a & c) | (b & c)
                else:
                    op = {"AND": np.bitwise_and, "OR": np.bitwise_or, "XOR": np.bitwise_xor}[f]
                    out = ins[0]
                    for x in ins[1:]:
                        out = op(out, x)
                sim[grp] = out
    return sim


def classes(code, edge_index, kind, batch=None, patterns=32768, seed=0, exhaustive=False, words_per_pass=None):
    """Functional equivalence classes on the simulated patterns: (rep int64 [N], complemented bool [N]).  Two nodes of
    one circuit share a class when their words are equal on every pattern, or one's are the bitwise NOT of the other's.
    A node's canonical words are its words when it is 0 on pattern 0 and their NOT otherwise; nodes are grouped by
    (circuit, canonical words), ``rep`` is the smallest node id of the group, and ``complemented[v]`` is True when v's
    value on pattern 0 differs from its representative's.  ``words_per_pass`` splits the words into passes."""
    net, patterns = _prepare(code, edge_index, kind, batch, patterns, exhaustive)
    n = net["n"]
    total = patterns // 64
    step = total if words_per_pass is None else int(words_per_pass)
    words = np.concatenate([pass_words(net, np.arange(first, min(first + step, total)), seed, exhaustive)
                            for first in range(0, total, step)], axis=1)
    bit0 = (words[:, 0] & np.uint64(1)).astype(bool)
    canon = np.where(bit0[:, None], ~words, words)
    key = np.concatenate([net["batch"].astype(np.uint64)[:, None], canon], axis=1)
    _, group = np.unique(key, axis=0, return_inverse=True)
    group = group.reshape(-1)
    first = np.full(group.max() + 1 if n else 0, n, np.int64)
    np.minimum.at(first, group, np.arange(n))
    rep = first[group]
    return rep, bit0 != bit0[rep]
