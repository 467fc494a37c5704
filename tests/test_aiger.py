"""AIGER netlists into circuit dicts (deepgate/aiger.py) and their labels.
CPU: ASCII and binary twins give identical dicts; every output and AND variable keeps its meaning, checked by evaluating the
file directly against the numpy simulator's words; adders and multipliers compute a + b and a * b; the four layouts parse
and level; write_npz -> NpzParser; every error names the file and the place; a 1-million-AND binary file converts.
GPU: exhaustive labels equal the direct evaluation as counts for all four kinds; a 200 k-AND sequential netlist goes
through ``python -m deepgate.simulate --aiger``, NpzParser and one training epoch."""
import os
import subprocess
import sys
import time

import numpy as np
import pytest
import torch

import sim_classes_oracle as SO

# ------------------------------------------------------------------ fixtures (ASCII, hand-written)
FIXTURES = {
    # constant fan-ins: 8 = AND(a, 1) = a, 10 = AND(8, 0) = 0, 12 = AND(NOT 10, b) = b, 14 = AND(12, NOT c);
    # outputs: 14, 10 (constant 0), 1 (constant 1), 13 (NOT b through an alias)
    "consts": "aag 7 3 0 4 4\n2\n4\n6\n14\n10\n1\n13\n8 2 1\n10 8 0\n12 11 4\n14 12 7\n",
    # AND(a, a) = a, AND(a, NOT a) = 0, then ANDs over them; complemented outputs
    "same": "aag 6 2 0 3 4\n2\n4\n12\n9\n7\n6 2 2\n8 2 3\n10 6 5\n12 10 7\n",
    # two latches (one with a reset value): current states are inputs, next states outputs
    "latches": "aag 7 2 2 2 3\n2\n4\n6 13\n8 10 1\n14\n7\n10 2 6\n12 10 9\n14 12 4\n",
    # bad-state and constraint sections
    "bc": "aag 5 2 0 1 3 1 1\n2\n4\n10\n7\n9\n6 2 4\n8 3 5\n10 7 9\n",
    # ANDs out of order (and inputs not numbered 2, 4, ...)
    "unordered": "aag 8 3 0 2 5\n10\n2\n16\n13\n9\n12 14 6\n6 2 11\n14 8 17\n8 10 2\n4 12 7\n",
    # a symbol table and comments
    "symbols": "aag 5 3 0 2 2\n2\n4\n6\n10\n11\n8 2 4\n10 8 7\ni0 a\ni1 b\ni2 c\no0 f\no1 nf\nc\nmade by hand\n8 2 4\n",
}


def parse_aag(text):
    """The test's own reading of an ASCII file: (I, L, O, B, C, inputs, latches [(lhs, next, reset)], outputs (all
    sections), ands [(lhs, rhs0, rhs1)], the text after the ANDs)."""
    lines = text.split("\n")
    M, I, L, O, A, B, C = (list(map(int, lines[0].split()[1:])) + [0, 0])[:7]
    k = 1
    inputs = [int(lines[k + j]) for j in range(I)]
    k += I
    latches = []
    for j in range(L):
        t = list(map(int, lines[k + j].split()))
        latches.append((t[0], t[1], t[2] if len(t) > 2 else 0))
    k += L
    outputs = [int(lines[k + j]) for j in range(O + B + C)]
    k += O + B + C
    ands = [tuple(map(int, lines[k + j].split())) for j in range(A)]
    return I, L, O, B, C, inputs, latches, outputs, ands, "\n".join(lines[k + A:])


def evaluate(text):
    """Direct AIGER semantics over every assignment of the I + L input variables (input j of primary inputs, then latch
    states, takes bit j of the pattern number): ``value(literal)`` -> bool [2^(I + L)], and the input count."""
    I, L, O, B, C, inputs, latches, outputs, ands, _ = parse_aag(text)
    k = I + L
    t = np.arange(1 << k)
    val = {0: np.zeros(1 << k, bool)}
    for j, lit in enumerate(inputs + [l[0] for l in latches]):
        val[lit >> 1] = (t >> j) & 1 == 1
    defs = {lhs >> 1: (a, b) for lhs, a, b in ands}

    def var(v):
        if v not in val:
            a, b = defs[v]
            val[v] = value(a) & value(b)
        return val[v]

    def value(lit):
        return var(lit >> 1) ^ bool(lit & 1)
    return value, k


def dfs_order(ands):
    """ANDs in file order, each after its not yet placed fan-in ANDs (depth-first, rhs0 first)."""
    defs = {lhs >> 1: (a, b) for lhs, a, b in ands}
    placed, order = set(), []

    def visit(v):
        if v in placed or v not in defs:
            return
        visit(defs[v][0] >> 1)
        visit(defs[v][1] >> 1)
        placed.add(v)
        order.append(v)
    for lhs, _, _ in ands:
        visit(lhs >> 1)
    return order


def encode_binary(I, latch_next, latch_reset, outputs, n_bc, ands, trailer=b""):
    """A binary AIGER file from arrays already in binary numbering: inputs 1..I, latches I+1..I+L, AND i has lhs
    2 (I + L + 1 + i); ``ands`` [A, 2] (rhs0, rhs1) in any order within a row; ``outputs`` are O then B then C literals
    with ``n_bc`` = (B, C)."""
    L, A = len(latch_next), len(ands)
    ands = np.sort(np.asarray(ands, np.int64).reshape(A, 2), axis=1)[:, ::-1]
    lhs = 2 * (I + L + 1 + np.arange(A, dtype=np.int64))
    d = np.stack([lhs - ands[:, 0], ands[:, 0] - ands[:, 1]], axis=1).reshape(-1).astype(np.uint64)
    nbytes = 1 + sum(((d >> np.uint64(7 * j)) > 0).astype(np.int64) for j in range(1, 10))
    k = np.arange(int(nbytes.sum())) - np.repeat(np.cumsum(nbytes) - nbytes, nbytes)
    dd = np.repeat(d, nbytes)
    more = np.where(k < np.repeat(nbytes, nbytes) - 1, 0x80, 0).astype(np.uint64)        # continuation bit
    byte = ((dd >> (7 * k).astype(np.uint64)) & np.uint64(0x7F)) | more
    B, C = n_bc
    head = "aig %d %d %d %d %d" % (I + L + A, I, L, len(outputs) - B - C, A) + (" %d %d" % (B, C) if B or C else "")
    rows = [head] + ["%d %d" % (n, r) if r else "%d" % n for n, r in zip(latch_next, latch_reset)] + ["%d" % o for o in outputs]
    return ("\n".join(rows) + "\n").encode() + byte.astype(np.uint8).tobytes() + trailer


def to_binary(text):
    """The binary twin of an ASCII file (variables renumbered, ANDs in dfs_order) and the map old variable -> new."""
    I, L, O, B, C, inputs, latches, outputs, ands, trailer = parse_aag(text)
    order = [lit >> 1 for lit in inputs] + [l[0] >> 1 for l in latches] + dfs_order(ands)
    new = {0: 0}
    new.update({v: j + 1 for j, v in enumerate(order)})
    ren = lambda lit: 2 * new[lit >> 1] + (lit & 1)                  # noqa: E731
    defs = {lhs >> 1: (a, b) for lhs, a, b in ands}
    rows = [(ren(defs[v][0]), ren(defs[v][1])) for v in dfs_order(ands)]
    data = encode_binary(I, [ren(l[1]) for l in latches], [l[2] if l[2] in (0, 1) else ren(l[2]) for l in latches],
                         [ren(o) for o in outputs], (B, C), np.array(rows, np.int64).reshape(-1, 2),
                         trailer.encode() if trailer.strip() else b"")
    return data, new


class Aag(object):
    """Builds an ASCII AIGER file gate by gate, without simplifying (constants and all)."""

    def __init__(self):
        self.m, self.inputs, self.ands, self.outputs = 0, [], [], []

    def input(self):
        self.m += 1
        self.inputs.append(2 * self.m)
        return 2 * self.m

    def AND(self, a, b):
        self.m += 1
        self.ands.append((2 * self.m, a, b))
        return 2 * self.m

    def OR(self, a, b):
        return self.AND(a ^ 1, b ^ 1) ^ 1

    def XOR(self, a, b):
        return self.OR(self.AND(a, b ^ 1), self.AND(a ^ 1, b))

    def full_add(self, a, b, c):
        p = self.XOR(a, b)
        return self.XOR(p, c), self.OR(self.AND(a, b), self.AND(p, c))

    def text(self):
        rows = ["aag %d %d 0 %d %d" % (self.m, len(self.inputs), len(self.outputs), len(self.ands))]
        rows += ["%d" % i for i in self.inputs] + ["%d" % o for o in self.outputs] + ["%d %d %d" % a for a in self.ands]
        return "\n".join(rows) + "\n"


def adder(n):
    """n-bit ripple-carry adder: inputs a0..a(n-1), b0..b(n-1); outputs the n + 1 bits of a + b (carry-in constant 0)."""
    g = Aag()
    a = [g.input() for _ in range(n)]
    b = [g.input() for _ in range(n)]
    c = 0
    for i in range(n):
        s, c = g.full_add(a[i], b[i], c)
        g.outputs.append(s)
    g.outputs.append(c)
    return g.text()


def multiplier(n):
    """n x n array multiplier: inputs a0..a(n-1), b0..b(n-1); outputs the 2n bits of a * b.  Rows of partial products
    are added with ripple-carry adders starting from constant 0."""
    g = Aag()
    a = [g.input() for _ in range(n)]
    b = [g.input() for _ in range(n)]
    acc = [0] * (2 * n)
    for j in range(n):
        c = 0
        for i in range(n):
            acc[i + j], c = g.full_add(acc[i + j], g.AND(a[i], b[j]), c)
        for k in range(i + j + 1, 2 * n):
            acc[k], c = g.full_add(acc[k], 0, c)
    g.outputs = acc
    return g.text()


def write(tmp_path, name, data):
    p = tmp_path / name
    p.write_bytes(data if isinstance(data, bytes) else data.encode())
    return str(p)


def read(path, kind="aig"):
    from deepgate.aiger import read_aiger
    return read_aiger(path, kind)


def node_words(c, kind):
    """Every node's value on every assignment of its inputs, by oracle/logic_sim.py's exhaustive simulation: bool [N, 2^K]."""
    net, patterns = SO._prepare(c["x"][:, 1], c["edge_index"].T, kind, None, 64, True)
    words = SO.pass_words(net, np.arange(patterns // 64), 0, True)
    bits = np.unpackbits(words.view(np.uint8), axis=1, bitorder="little").astype(bool)
    k = int((c["x"][:, 1] == 0).sum())
    return bits[:, :1 << k]


def literal_bits(c, words, lit, need_not_node=False):
    """Value of a node-space literal (``2 node + complemented``, node -1 the constant) from the node words; a complemented
    literal is read from its NOT node when there is one (required when ``need_not_node``)."""
    if lit < 0:
        return np.full(words.shape[1], bool(lit & 1))
    n = lit >> 1
    if not lit & 1:
        return words[n]
    ei = c["edge_index"]
    not_code = 2                                           # NOT in every code table
    nots = ei[(ei[:, 0] == n) & (c["x"][ei[:, 1], 1] == not_code), 1]
    assert nots.size <= 1, "NOT node of %d is not shared" % n
    if need_not_node:
        assert nots.size == 1, "complemented output on node %d has no NOT node" % n
    return words[nots[0]] if nots.size else ~words[n]


def expected_node_bits(c, value):
    """Every node's value from the direct evaluation of the file: an INPUT or AND node is the variable that maps to it in
    ``lit``, a NOT node the complement of its predecessor."""
    lit, x, ei = c["lit"], c["x"], c["edge_index"]
    out = [None] * len(x)
    var_of = {int(l) >> 1: v for v, l in enumerate(lit) if l >= 0 and not l & 1 and v > 0}
    for node in range(len(x)):
        if x[node, 1] == 2:
            pred = ei[ei[:, 1] == node, 0]
            assert pred.size == 1
            out[node] = ~out[int(pred[0])]
        else:
            out[node] = value(2 * var_of[node])
    return np.array(out)


def assert_meaning(c, text, kind="aig"):
    """Every output and every AND variable of the file, evaluated directly, equals the simulated node that represents it."""
    value, k = evaluate(text)
    I, L, O, B, C, inputs, latches, outputs, ands, _ = parse_aag(text)
    words = node_words(c, kind)
    assert words.shape[1] == 1 << k
    outs = outputs[:O] + [l[1] for l in latches] + outputs[O:]
    assert len(c["outputs"]) == len(outs)
    for lit, got in zip(outs, c["outputs"]):
        assert np.array_equal(literal_bits(c, words, int(got), need_not_node=True), value(lit)), lit
    for lhs, _, _ in ands:
        assert np.array_equal(literal_bits(c, words, int(c["lit"][lhs >> 1])), value(lhs)), lhs
    assert np.array_equal(expected_node_bits(c, value), words)


def assert_same(a, b, var_map=None):
    for key in ("x", "edge_index", "outputs"):
        assert np.array_equal(a[key], b[key]), key
    assert a["name"] == b["name"]
    if var_map is None:
        assert np.array_equal(a["lit"], b["lit"])
    else:
        for old, new in var_map.items():
            assert a["lit"][old] == b["lit"][new], old


# ------------------------------------------------------------------ CPU
@pytest.mark.parametrize("name", sorted(FIXTURES))
def test_ascii_and_binary_give_identical_dicts(tmp_path, name):
    text = FIXTURES[name]
    data, var_map = to_binary(text)
    a = read(write(tmp_path, name + ".aag", text))
    (tmp_path / "bin").mkdir()
    b = read(write(tmp_path / "bin", name + ".aig", data))
    assert_same(a, b, var_map)


@pytest.mark.parametrize("name", sorted(FIXTURES))
def test_fixture_meaning_is_preserved(tmp_path, name):
    text = FIXTURES[name]
    c = read(write(tmp_path, name + ".aag", text))
    assert_meaning(c, text)
    code, ei = c["x"][:, 1], c["edge_index"]
    indeg = np.bincount(ei[:, 1], minlength=len(code))
    assert np.all(indeg[code == 1] == 2) and np.all(indeg[code == 2] == 1) and np.all(indeg[code == 0] == 0)
    assert np.all(ei[:, 0] < ei[:, 1])                       # node ids are a topological order
    ands = ei[code[ei[:, 1]] == 1]
    assert len({tuple(p) for p in ands}) == len(ands)        # distinct predecessors


def test_folding_and_node_order(tmp_path):
    c = read(write(tmp_path, "consts.aag", FIXTURES["consts"]))
    # inputs a b c, NOT c, then the only AND left, AND(b, NOT c), and NOT b for output 13
    assert c["x"][:, 1].tolist() == [0, 0, 0, 2, 2, 1]
    assert c["edge_index"].tolist() == [[1, 3], [2, 4], [1, 5], [4, 5]]
    assert c["outputs"].tolist() == [10, -2, -1, 3]
    assert c["lit"].tolist() == [-2, 0, 2, 4, 0, -2, 2, 10]
    s = read(write(tmp_path, "same.aag", FIXTURES["same"]))
    assert s["lit"][3] == 0 and s["lit"][4] == -2            # AND(a, a) = a, AND(a, NOT a) = 0
    assert s["outputs"].tolist()[1:] == [-1, 1]
    lat = read(write(tmp_path, "latches.aag", FIXTURES["latches"]))
    assert lat["x"][:4, 1].tolist() == [0, 0, 0, 0] and lat["lit"][3] == 4 and lat["lit"][4] == 6
    u = read(write(tmp_path, "unordered.aag", FIXTURES["unordered"]))
    assert u["lit"][5] == 0 and u["lit"][1] == 2 and u["lit"][8] == 4      # inputs in file order: 10, 2, 16


@pytest.mark.parametrize("circuit,n", [("adder", 6), ("multiplier", 6), ("multiplier", 3)])
@pytest.mark.parametrize("form", ["aag", "aig"])
def test_arithmetic(tmp_path, circuit, n, form):
    text = adder(n) if circuit == "adder" else multiplier(n)
    path = write(tmp_path, "%s%d.%s" % (circuit, n, form), text if form == "aag" else to_binary(text)[0])
    c = read(path, "xag")
    words = node_words(c, "xag")
    t = np.arange(1 << (2 * n))
    a, b = t & ((1 << n) - 1), t >> n
    got = sum(literal_bits(c, words, int(o), need_not_node=True).astype(np.int64) << j for j, o in enumerate(c["outputs"]))
    assert np.array_equal(got, a + b if circuit == "adder" else a * b)
    assert (c["outputs"] >= 0).all()
    if form == "aag":
        assert_meaning(c, text, "xag")


@pytest.mark.parametrize("kind", ["aig", "mig", "xmg", "xag"])
def test_layouts_parse_and_level(tmp_path, kind):
    from deepgate.parser_func_others import parse_pyg_mlpgate
    from deepgate.simulate import CODE_TABLES
    from deepgate.utils.dag_utils import top_sort_host
    table = CODE_TABLES[kind]
    for name, text in sorted(FIXTURES.items()) + [("mult4", multiplier(4))]:
        c = read(write(tmp_path, name + ".aag", text), kind)
        code = c["x"][:, 1]
        assert set(code.tolist()) <= {table.index("INPUT"), table.index("AND"), table.index("NOT")}
        n = len(code)
        g = parse_pyg_mlpgate(c["x"], c["edge_index"], np.zeros(n, np.float32), np.zeros(1, np.float32),
                              np.zeros((1, 2), np.int64))
        level = top_sort_host(c["edge_index"].T, n).numpy()
        assert np.array_equal(g.forward_level.numpy(), level)
        src, dst = c["edge_index"].T
        assert np.all(level[dst] > level[src]) and np.all(level[code == 0] == 0)
    a = read(write(tmp_path, "m.aag", multiplier(4)), "aig")
    m = read(str(tmp_path / "m.aag"), kind)
    assert np.array_equal(a["edge_index"], m["edge_index"])
    assert np.array_equal(a["x"][:, 1] == 1, m["x"][:, 1] == table.index("AND"))


@pytest.mark.parametrize("kind", ["aig", "mig"])
def test_write_npz_round_trips_through_npz_parser(tmp_path, kind):
    import deepgate
    from deepgate.aiger import read_aiger_files
    d = tmp_path / "netlists"
    d.mkdir()
    for name, text in FIXTURES.items():
        write(d, name + ".aag", text)
    write(d, "adder4.aig", to_binary(adder(4))[0])
    write(d, "notes.txt", "not a netlist")
    circuits = read_aiger_files([str(d), write(tmp_path, "mult3.aag", multiplier(3))], kind)
    assert [c["name"] for c in circuits] == ["adder4", "bc", "consts", "latches", "same", "symbols", "unordered", "mult3"]
    for i, c in enumerate(circuits):
        n = len(c["x"])
        c["prob"] = np.random.default_rng(i).random(n).astype(np.float32)
        c["tt_pair_index"] = np.random.default_rng(i).integers(0, n, (5, 2))
        c["tt_sim"] = np.random.default_rng(50 + i).random(5).astype(np.float32)
    root = str(tmp_path / "ds")
    os.makedirs(root)
    gp, lp = deepgate.write_npz(circuits, os.path.join(root, "graphs.npz"),
                                None if kind == "aig" else os.path.join(root, "labels.npz"), kind)
    graphs = deepgate.NpzParser(root, gp, lp, kind, random_shuffle=False, trainval_split=1.0).train_dataset.graphs
    assert [g.name for g in graphs] == [c["name"] for c in circuits]
    for c, g in zip(circuits, graphs):
        assert torch.equal(g.edge_index, torch.from_numpy(c["edge_index"].T.copy()))
        assert torch.equal(g.gate.reshape(-1).long(), torch.from_numpy(c["x"][:, 1]))
        assert torch.equal(g.prob.reshape(-1), torch.from_numpy(c["prob"]))
        assert torch.equal(g.tt_sim, torch.from_numpy(c["tt_sim"]))
    with pytest.raises(ValueError, match="already read"):
        read_aiger_files([str(d), write(tmp_path, "bc.aag", FIXTURES["bc"])], kind)


def bin_file(head, lines, deltas):
    return (head + "\n" + "".join(l + "\n" for l in lines)).encode() + bytes(deltas)


ERRORS = [  # (file name, content, message after "<path>: ")
    ("extra_and.aag", "aag 3 2 0 1 1\n2\n4\n6\n6 2 4\n6 4 2\n", "line 6: expected the symbol table"),
    ("bad_m.aig", bin_file("aig 4 2 0 1 1", ["6"], [2, 2]), "line 1: a binary header needs M = I \\+ L \\+ A"),
    ("big.aag", "aag 3 2 0 1 1\n2\n4\n9\n6 2 4\n", "line 4: literal 9 is above 2M \\+ 1 = 7"),
    ("big_and.aag", "aag 3 2 0 1 1\n2\n4\n6\n6 2 8\n", "line 5: literal 8 is above"),
    ("odd_input.aag", "aag 3 2 0 1 1\n3\n4\n6\n6 2 4\n", "line 2: the input literal 3 must be even"),
    ("odd_latch.aag", "aag 3 1 1 1 1\n2\n5 6\n6\n6 2 4\n", "line 3: the latch literal 5 must be even"),
    ("odd_and.aag", "aag 3 2 0 1 1\n2\n4\n6\n7 2 4\n", "line 5: the AND literal 7 must be even"),
    ("twice.aag", "aag 3 2 0 1 2\n2\n4\n6\n6 2 4\n4 2 3\n", "line 6: variable 2 is defined twice"),
    ("undefined.aag", "aag 4 2 0 1 1\n2\n4\n6\n6 2 8\n", "line 5: variable 4 is used but never defined"),
    ("undefined_out.aag", "aag 4 2 0 1 1\n2\n4\n8\n6 2 4\n", "line 4: variable 4 is used but never defined"),
    ("cycle.aag", "aag 4 1 0 1 2\n2\n6\n6 2 8\n8 6 2\n", "line 5: combinational cycle"),
    ("order.aig", bin_file("aig 3 2 0 1 1", ["6"], [0, 2]), "byte 16: AND 0 breaks lhs > rhs0 >= rhs1"),
    ("order2.aig", bin_file("aig 4 2 0 1 2", ["8"], [2, 2, 3, 6]), "byte 18: AND 1 breaks lhs > rhs0 >= rhs1"),
    ("short.aag", "aag 3 2 0 1 1\n2\n4\n6\n", "line 5: file truncated: 1 AND lines expected from line 5"),
    ("short.aig", bin_file("aig 4 2 0 1 2", ["8"], [2, 2, 0x81]), "byte 19: file truncated: 4 AND deltas expected, 2"),
    ("short_outputs.aig", b"aig 3 2 0 2 1\n6\n", "line 3: file truncated: 2 output lines expected from line 2"),
    ("justice.aag", "aag 3 2 0 1 1 0 0 1 0\n2\n4\n6\n6 2 4\n", "line 1: justice \\(J = 1\\)"),
    ("not_aiger.aag", "aig x\n", "line 1: not an AIGER header"),
    ("word.aag", "aag 3 2 0 1 1\n2\n4\n6\n6 2 x\n", "line 5: not a literal"),
    ("width.aag", "aag 3 2 0 1 1\n2\n4\n6\n6 2\n", "line 5: expected 3 numbers on this AND line, found 2"),
]


@pytest.mark.parametrize("case", range(len(ERRORS)))
def test_errors_name_the_file_and_place(tmp_path, case):
    import re
    name, data, msg = ERRORS[case]
    path = write(tmp_path, name, data)
    with pytest.raises(ValueError, match="^" + re.escape(path) + ": " + msg):
        read(path)
    with pytest.raises(ValueError, match="kind"):
        read(path, "nand")


def random_aig(I, L, A, window, seed, n_out=32):
    """A random binary AIGER file: AND i draws two distinct fan-in variables among the ``window`` variables before it,
    each complemented with probability 1/2; latches take random next-state literals, outputs are the last ANDs.
    Returns (bytes, A)."""
    rng = np.random.default_rng(seed)
    v = I + L + 1 + np.arange(A, dtype=np.int64)
    lo = np.maximum(1, v - window)
    span = v - lo
    f0 = lo + (rng.random(A) * span).astype(np.int64)
    f1 = lo + (f0 - lo + 1 + (rng.random(A) * (span - 1)).astype(np.int64)) % span
    ands = np.stack([2 * f0 + rng.integers(0, 2, A), 2 * f1 + rng.integers(0, 2, A)], axis=1)
    M = I + L + A
    nxt = 2 + rng.integers(0, 2 * M, L)
    outs = 2 * v[-n_out:] + rng.integers(0, 2, n_out)
    return encode_binary(I, nxt.tolist(), [0] * L, outs.tolist(), (0, 0), ands), A


def test_million_and_binary_converts(tmp_path):
    data, A = random_aig(64, 64, 1_000_000, 2000, seed=1)
    path = write(tmp_path, "big.aig", data)
    t = time.perf_counter()
    c = read(path)
    dt = time.perf_counter() - t
    code = c["x"][:, 1]
    assert (code == 0).sum() == 128 and (code == 1).sum() == A
    assert np.all(c["edge_index"][:, 0] < c["edge_index"][:, 1])
    print("1 000 000 ANDs: %.2f s on the host" % dt)


def test_cli_aiger_arguments(tmp_path):
    from deepgate.simulate import main
    with pytest.raises(SystemExit):                          # one input source
        main(["--graphs", "g.npz", "--aiger", "a.aag", "--type", "aig", "--out", "d"])
    with pytest.raises(SystemExit):
        main(["--type", "aig", "--out", "d"])
    bad = write(tmp_path, "cycle.aag", ERRORS[10][1])
    with pytest.raises(ValueError, match="cycle.aag: line 5"):
        main(["--aiger", bad, "--type", "aig", "--out", str(tmp_path / "o")])


# ------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["aig", "mig", "xmg", "xag"])
def test_exhaustive_labels_equal_direct_evaluation(tmp_path, kind):
    import deepgate
    texts = dict(FIXTURES, adder6=adder(6), mult6=multiplier(6), mult3=multiplier(3))
    circuits, values = [], []
    for name, text in sorted(texts.items()):
        circuits.append(read(write(tmp_path, name + ".aag", text), kind))
        values.append(evaluate(text))
    labelled = deepgate.label_circuits(circuits, kind, "cuda:0", exhaustive=True)
    patterns = max(64, 1 << max(k for _, k in values))
    for c, (value, k) in zip(labelled, values):
        want = expected_node_bits(c, value).sum(axis=1) * (patterns >> k)
        got = c["prob"].astype(np.float64) * patterns
        assert np.array_equal(got, want.astype(np.float64)), c["name"]


@pytest.mark.gpu
def test_sequential_netlist_cli_to_training(tmp_path):
    import types
    import deepgate
    d = tmp_path / "netlists"
    d.mkdir()
    data, A = random_aig(64, 512, 200_000, 800, seed=3)
    write(d, "seq200k.aig", data)
    for i in range(3):                                       # read after it, in name order: training needs a val set
        write(d, "small%d.aig" % i, random_aig(8, 4, 300, 50, seed=4 + i, n_out=8)[0])
    write(d, "consts.aag", FIXTURES["consts"])              # read first; two of its outputs are constants
    out = tmp_path / "ds"
    env = dict(os.environ)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env["PYTHONPATH"] = os.pathsep.join([os.path.join(root, "multi-gate-vae_b200"), env.get("PYTHONPATH", "")])
    r = subprocess.run([sys.executable, "-m", "deepgate.simulate", "--aiger", str(d), "--type", "mig", "--out", str(out),
                        "--class-pairs", "16"], env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "dropped 2 outputs that fold to constants" in r.stdout and "labelled 5 circuits" in r.stdout
    torch.manual_seed(0)
    parser = deepgate.NpzParser(str(out), str(out / "graphs.npz"), str(out / "labels.npz"), "mig", random_shuffle=False,
                                trainval_split=0.5)
    train, val = parser.get_dataset()
    g = train[1]
    assert train[0].name == "consts" and g.name == "seq200k" and len(val) == 3
    assert int((g.gate == 0).sum()) == 64 + 512 and int((g.gate == 3).sum()) == A
    assert int(g.forward_level.max()) + 1 > 1000
    assert g.tt_pair_index.shape == (2, 64) and torch.all((g.prob >= 0) & (g.prob <= 1))
    enc = deepgate.digae_layer.DirectMultiGCNEncoder(dim_hidden=64, dim_feature=6, s_rounds=1, t_rounds=1)
    model = deepgate.dg_ae_model_mig.Model(struct_encoder=enc, dim_hidden=64)
    args = types.SimpleNamespace(model="DG_AE", type="mig")
    trainer = deepgate.Trainer(args, model, training_id="aiger", save_dir=str(tmp_path / "exp"), device="cuda:0",
                               batch_size=1, distributed=False, rc_prob_func_weight=[1.0, 4.0, 4.0])
    trainer.train(1, train, val)
    log = open(trainer.log_path).read()
    assert "train|" in log and "nan" not in log.lower()
