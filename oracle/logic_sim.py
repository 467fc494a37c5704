"""Reference bit-parallel logic simulator in numpy: what the tests trust for deepgate.simulate.

Same definitions as csrc/logic_sim.cu (include/mgv_b200.h, "logic simulation"):
  * gate functions by code: AIG {0 INPUT, 1 AND, 2 NOT}; MIG / XMG / XAG {0 INPUT, 1 MAJ, 2 NOT, 3 AND, 4 OR, 5 XOR};
    AND / OR / XOR reduce over all predecessors;
  * 64 patterns per uint64 word.  Random mode: word w of an INPUT = mix(mix(seed) ^ (rank << 40 | w)), mix = the
    splitmix64 finaliser, rank = the INPUT's position among the INPUTs of its own circuit.  Exhaustive mode: pattern
    t = 64 w + bit, the INPUT takes bit rank of t;
  * counts: ones[v] = patterns where node v is 1, diff[p] = patterns where the two nodes of pair p differ.
Kept plain: one topological level at a time, one gate function at a time.
"""
import numpy as np

CODE_TABLES = {
    "aig": {0: "INPUT", 1: "AND", 2: "NOT"},
    "mig": {0: "INPUT", 1: "MAJ", 2: "NOT", 3: "AND", 4: "OR", 5: "XOR"},
}
for _k in ("xmg", "xag"):
    CODE_TABLES[_k] = CODE_TABLES["mig"]

M64 = np.uint64(0xFFFFFFFFFFFFFFFF)


def mix(z):
    """splitmix64 finaliser on a uint64 array (wrapping arithmetic)."""
    z = np.asarray(z, dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = z + np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def popcount(a):
    """Set bits per row of a uint64 array [..., W] -> int64 [...]."""
    b = np.ascontiguousarray(a).view(np.uint8)
    return np.unpackbits(b, axis=-1).sum(axis=-1, dtype=np.int64)


def levels(edge_index, n):
    """ASAP level of every node (0 = no predecessor), by peeling in-degree-zero frontiers."""
    src, dst = np.asarray(edge_index[0], np.int64), np.asarray(edge_index[1], np.int64)
    indeg = np.bincount(dst, minlength=n)
    by_src = np.argsort(src, kind="stable")
    out_ptr = np.zeros(n + 1, np.int64)
    np.cumsum(np.bincount(src, minlength=n), out=out_ptr[1:])
    out_dst = dst[by_src]
    level = np.full(n, -1, np.int64)
    frontier = np.flatnonzero(indeg == 0)
    lvl = 0
    while frontier.size:
        level[frontier] = lvl
        succ = np.concatenate([out_dst[out_ptr[v]:out_ptr[v + 1]] for v in frontier]) if frontier.size else frontier
        np.subtract.at(indeg, succ, 1)
        frontier = np.unique(succ[indeg[succ] == 0])
        lvl += 1
    if (level < 0).any():
        raise ValueError("the graph has a cycle")
    return level


def input_ranks(code, batch):
    """Position of every INPUT among the INPUTs of its own circuit (-1 elsewhere)."""
    rank = np.full(code.size, -1, np.int64)
    for c in np.unique(batch):
        idx = np.flatnonzero((batch == c) & (code == 0))
        rank[idx] = np.arange(idx.size)
    return rank


def input_words(rank, words, seed, exhaustive):
    """uint64 [len(rank), len(words)] words of the INPUTs with the given ranks."""
    rank = np.asarray(rank, np.uint64)[:, None]
    w = np.asarray(words, np.uint64)[None, :]
    if not exhaustive:
        return mix(mix(np.uint64(seed)) ^ ((rank << np.uint64(40)) | w))
    bit = np.arange(64, dtype=np.uint64)
    t = (w[..., None] << np.uint64(6)) | bit                          # [1, W, 64] pattern numbers
    on = (t >> rank[..., None]) & np.uint64(1)                         # [R, W, 64]
    return (on << bit).sum(axis=-1, dtype=np.uint64)


def simulate(code, edge_index, kind, batch=None, pairs=None, patterns=32768, seed=0, exhaustive=False, words_per_pass=None):
    """Returns (ones int64 [N], diff int64 [P], patterns).  ``edge_index`` [2, E] (row 0 = source); ``batch`` [N] circuit
    of each node (None: one circuit); ``pairs`` [2, P]; ``words_per_pass`` splits the words into passes (counts add up)."""
    code = np.asarray(code, np.int64).reshape(-1)
    n = code.size
    ei = np.asarray(edge_index, np.int64).reshape(2, -1)
    batch = np.zeros(n, np.int64) if batch is None else np.asarray(batch, np.int64)
    pairs = np.zeros((2, 0), np.int64) if pairs is None else np.asarray(pairs, np.int64).reshape(2, -1)
    table = CODE_TABLES[kind]
    fn = np.array([table.get(int(c), "NONE") for c in code])
    if (fn == "NONE").any():
        raise ValueError("undefined gate code at node %d" % int(np.flatnonzero(fn == "NONE")[0]))
    rank = input_ranks(code, batch)
    if exhaustive:
        k = int(np.bincount(batch[code == 0]).max()) if (code == 0).any() else 0
        if k > 24:
            raise ValueError("exhaustive simulation of %d inputs" % k)
        patterns = max(64, 1 << k)
    if patterns <= 0 or patterns % 64:
        raise ValueError("patterns must be a positive multiple of 64")
    total = patterns // 64
    step = total if words_per_pass is None else int(words_per_pass)
    lvl = levels(ei, n)
    order = np.argsort(ei[1], kind="stable")                         # predecessors by node, ascending edge id
    preds_src, in_deg = ei[0][order], np.bincount(ei[1], minlength=n)
    in_ptr = np.zeros(n + 1, np.int64)
    np.cumsum(in_deg, out=in_ptr[1:])
    ones = np.zeros(n, np.int64)
    diff = np.zeros(pairs.shape[1], np.int64)
    for first in range(0, total, step):
        words = np.arange(first, min(first + step, total))
        sim = np.zeros((n, words.size), np.uint64)
        for l in range(int(lvl.max()) + 1 if n else 0):
            at = lvl == l
            for f in np.unique(fn[at]):
                nodes = np.flatnonzero(at & (fn == f))
                if f == "INPUT":
                    sim[nodes] = input_words(rank[nodes], words, seed, exhaustive)
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
        ones += popcount(sim)
        if pairs.shape[1]:
            diff += popcount(sim[pairs[0]] ^ sim[pairs[1]])
    return ones, diff, patterns
