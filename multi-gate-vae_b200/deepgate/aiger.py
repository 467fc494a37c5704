"""Read AIGER netlists (ASCII ``.aag`` and binary ``.aig``, AIGER 1.9) into the circuit dicts that ``label_circuits`` and
``write_npz`` take, so that public benchmark circuits can be labelled and trained on.

    c = read_aiger("adder.aig", "aig")                       # one circuit dict
    circuits = read_aiger_files(["bench/", "mult.aag"], "mig")   # files, and the .aag / .aig files of directories
    python -m deepgate.simulate --aiger bench/ --type mig --out DIR

The result is the combinational core of the netlist in the reference's circuit shape: explicit NOT nodes and ANDs of
fan-in 2 over distinct predecessors, with no constant node.
  * Node order: primary inputs, then latch inputs (both in file order), then the NOT nodes of those inputs (same order),
    then the ANDs in topological order, each directly followed by its NOT node if it has one.  The ANDs keep the file's
    order when that is topological (always so in a binary file); otherwise every AND is preceded by those of its fan-in
    ANDs not placed yet, depth-first, rhs0 first.
  * NOT nodes: one per variable whose complemented literal is used as a fan-in of a kept AND or as an output, shared by
    every such use.
  * Constants are folded: AND(x, 0) = 0, AND(x, 1) = x, AND(a, a) = a, AND(a, NOT a) = 0, through the whole graph.  An AND
    that folds to a constant or to another literal is an alias, not a node; an output that folds to a constant gets no node.
  * Latches are cut: each latch's current-state variable becomes an INPUT node and its next-state literal is treated as an
    output.  Reset values are read and ignored, so a node fed by a latch is labelled from random (or exhaustive) input
    patterns like any other input.  Bad-state (B) and constraint (C) literals are outputs too; justice (J) and fairness
    (F) properties are rejected.  The symbol table and the comment section are skipped.
Gate codes come from ``simulate.CODE_TABLES``: ``aig`` INPUT 0, AND 1, NOT 2; ``mig`` / ``xmg`` / ``xag`` INPUT 0, NOT 2,
AND 3 (an AIG is a valid circuit of each kind, emitted as is).

Besides ``x`` [N, 2] (node id, gate code), ``edge_index`` [E, 2] (src, dst; sorted by dst, then src) and ``name`` (the
file stem), a dict carries ``lit`` int64 [M + 1] and ``outputs`` int64 [O + L + B + C]: the function of every AIGER
variable and of every output literal (primary outputs, latch next states, bad states, constraints, in file order) as a
literal over the nodes, ``2 * node + complemented``, where node -1 is the constant 0 (so -2 = 0, -1 = 1).  A variable
that is neither defined nor used reads -2.  A malformed file raises ``ValueError`` naming the file and the line or byte.
"""
import os

import numpy as np

from .simulate import CODE_TABLES

SUFFIXES = (".aag", ".aig")


class _Src(object):
    """Error messages that name the file and a place in it."""

    def __init__(self, path):
        self.path = str(path)

    def error(self, where, msg):
        return ValueError("%s: %s: %s" % (self.path, where, msg))


def _rows(src, lines, first, count, widths, what):
    """int64 [count, max(widths)] from ``count`` lines starting at index ``first`` of ``lines`` (line ``first + 1`` of
    the file); a line has one of ``widths`` tokens, missing trailing ones read -1."""
    if first + count > len(lines):
        raise src.error("line %d" % (len(lines) + 1), "file truncated: %d %s lines expected from line %d"
                        % (count, what, first + 1))
    rows = [ln.split() for ln in lines[first:first + count]]
    w = max(widths)
    lens = np.fromiter((len(r) for r in rows), np.int64, count)
    bad = np.flatnonzero(~np.isin(lens, widths))
    if bad.size:
        raise src.error("line %d" % (first + 1 + bad[0]), "expected %s numbers on this %s line, found %d"
                        % (" or ".join(map(str, widths)), what, lens[bad[0]]))
    if (lens != w).any():
        rows = [r + [b"-1"] * (w - len(r)) for r in rows]
    try:
        out = np.array(rows, dtype=np.int64).reshape(count, w)
    except (ValueError, OverflowError):
        out = None
    if out is None or (out[lens[:, None] > np.arange(w)] < 0).any():
        for k, r in enumerate(rows):
            if not all(t.isdigit() and len(t) <= 18 for t in r[:lens[k]]):
                raise src.error("line %d" % (first + 1 + k), "not a literal: %r" % b" ".join(r[:lens[k]]))
    return out


def _header(src, line):
    tok = line.split()
    if len(tok) < 6 or len(tok) > 10 or tok[0] not in (b"aag", b"aig") or not all(t.isdigit() for t in tok[1:]):
        raise src.error("line 1", "not an AIGER header 'aag|aig M I L O A [B C J F]': %r" % line[:80])
    h = [int(t) for t in tok[1:]] + [0] * (10 - len(tok))
    if h[7] or h[8]:
        raise src.error("line 1", "justice (J = %d) and fairness (F = %d) properties are not supported" % (h[7], h[8]))
    return tok[0] == b"aig", h[:7]


def _varints(src, buf, base, count):
    """The first ``count`` unsigned LEB128 numbers of ``buf`` (byte ``base`` of the file on): (int64 [count], byte offset
    of each number in ``buf``, bytes used)."""
    b = np.frombuffer(buf, np.uint8)
    ends = np.flatnonzero(b < 0x80)[:count]
    if ends.size < count:
        raise src.error("byte %d" % (base + b.size), "file truncated: %d AND deltas expected, %d found" % (count, ends.size))
    starts = np.zeros(count, np.int64)
    starts[1:] = ends[:-1] + 1
    length = ends - starts + 1
    if count and length.max() > 9:
        k = int(np.argmax(length > 9))
        raise src.error("byte %d" % (base + starts[k]), "a delta longer than 9 bytes")
    used = int(ends[-1]) + 1 if count else 0
    shift = ((np.arange(used) - np.repeat(starts, length)) * 7).astype(np.uint64)
    vals = np.add.reduceat((b[:used] & 0x7F).astype(np.uint64) << shift, starts) if count else np.zeros(0, np.uint64)
    return vals.astype(np.int64), starts, used


def _parse(src, data):
    """The netlist as literal arrays: M, O, inputs [I], latches [L, 2] (lhs, next), outputs [O + B + C], ands [A, 3], and
    ``where(section, index)``, the place of an entry for error messages."""
    nl = data.find(b"\n")
    binary, (M, I, L, O, A, B, C) = _header(src, data if nl < 0 else data[:nl])
    n_out = O + B + C
    if not binary:
        lines = data.split(b"\n")                               # lines[k] is line k + 1 of the file
        if lines[-1] == b"":
            lines.pop()
        inputs = _rows(src, lines, 1, I, (1,), "input")[:, 0]
        lat = _rows(src, lines, 1 + I, L, (2, 3), "latch")[:, :2]
        outs = _rows(src, lines, 1 + I + L, n_out, (1,), "output")[:, 0]
        ands = _rows(src, lines, 1 + I + L + n_out, A, (3,), "AND")
        after = 1 + I + L + n_out + A
        tail, tail_where = (lines[after][:1] if after < len(lines) else b""), "line %d" % (after + 1)

        def where(section, k):
            return "line %d" % (2 + k + {"input": 0, "latch": I, "output": I + L, "and": I + L + n_out}[section])
    else:
        if M != I + L + A:
            raise src.error("line 1", "a binary header needs M = I + L + A, got M = %d, I + L + A = %d" % (M, I + L + A))
        lines = data.split(b"\n", 1 + L + n_out)
        rest = lines.pop() if len(lines) > 1 + L + n_out else b""
        if rest == b"" and lines[-1] == b"":                     # the newline that ends the file
            lines.pop()
        lat = _rows(src, lines, 1, L, (1, 2), "latch")
        lat = np.stack([2 * (I + 1 + np.arange(L, dtype=np.int64)), lat[:, 0]], axis=1)
        outs = _rows(src, lines, 1 + L, n_out, (1,), "output")[:, 0]
        inputs = 2 * (1 + np.arange(I, dtype=np.int64))
        base = len(data) - len(rest)                            # file offset of the AND deltas
        d, starts, used = _varints(src, rest, base, 2 * A)
        lhs = 2 * (I + L + 1 + np.arange(A, dtype=np.int64))
        r0 = lhs - d[0::2]
        r1 = r0 - d[1::2]
        bad = np.flatnonzero((d[0::2] == 0) | (r1 < 0))
        if bad.size:
            k = int(bad[0])
            raise src.error("byte %d" % (base + starts[2 * k]), "AND %d breaks lhs > rhs0 >= rhs1 (lhs %d, deltas %d %d)"
                            % (k, lhs[k], d[2 * k], d[2 * k + 1]))
        ands = np.stack([lhs, r0, r1], axis=1)
        tail, tail_where = rest[used:used + 1], "byte %d" % (base + used)

        def where(section, k):
            if section == "and":
                return "byte %d" % (base + starts[2 * k])
            return "line %d" % (2 + k + (0 if section == "latch" else L))
    if tail not in (b"", b"\n", b"i", b"l", b"o", b"b", b"c", b"j", b"f"):
        raise src.error(tail_where, "expected the symbol table or the comment section after the %d ANDs the header "
                                    "declares" % A)
    return M, O, inputs, lat, outs, ands, where


def _check(src, M, inputs, lat, outs, ands, where):
    """Literal bounds, definitions and uses; returns the index in ``ands`` of every variable's defining AND (-1: none)."""
    uses = (("latch", lat[:, 1]), ("output", outs), ("and", ands[:, 1]), ("and", ands[:, 2]))
    defs = (("input", inputs), ("latch", lat[:, 0]), ("and", ands[:, 0]))
    for section, a in defs + uses:
        bad = np.flatnonzero(a > 2 * M + 1)
        if bad.size:
            raise src.error(where(section, int(bad[0])), "literal %d is above 2M + 1 = %d" % (a[bad[0]], 2 * M + 1))
    for section, a in defs:
        bad = np.flatnonzero((a & 1) | (a < 2))
        if bad.size:
            raise src.error(where(section, int(bad[0])), "the %s literal %d must be even and not 0"
                            % ("AND" if section == "and" else section, a[bad[0]]))
    var = np.concatenate([a for _, a in defs]) >> 1
    sec = np.repeat(np.arange(3), [a.size for _, a in defs])
    off = np.concatenate([np.arange(a.size) for _, a in defs])
    order = np.argsort(var, kind="stable")
    dup = order[1:][var[order[1:]] == var[order[:-1]]]
    if dup.size:
        k = int(dup.min())                                    # the first redefinition in file order
        raise src.error(where(defs[sec[k]][0], int(off[k])), "variable %d is defined twice" % var[k])
    defined = np.zeros(M + 1, bool)
    defined[0] = True                                         # the constant
    defined[var] = True
    for section, a in uses:
        bad = np.flatnonzero(~defined[a >> 1])
        if bad.size:
            raise src.error(where(section, int(bad[0])), "variable %d is used but never defined" % (a[bad[0]] >> 1))
    pos = np.full(M + 1, -1, np.int64)
    pos[ands[:, 0] >> 1] = np.arange(len(ands))
    return pos


def _topo_order(src, ands, pos, where):
    """Indices of ``ands`` in topological order: the file's order when it is one, else depth-first as the module says."""
    A = len(ands)
    kid = np.stack([pos[ands[:, 1] >> 1], pos[ands[:, 2] >> 1]], axis=1)
    if (kid < np.arange(A)[:, None]).all():
        return np.arange(A)
    kid = kid.tolist()
    state = bytearray(A)                                      # 0 new, 1 on the depth-first path, 2 placed
    order = []
    for root in range(A):
        stack = [root]
        while stack:
            i = stack[-1]
            if state[i] == 0:
                state[i] = 1
                for k in (kid[i][1], kid[i][0]):              # pushed last, expanded first: rhs0
                    if k >= 0 and state[k] == 1:
                        raise src.error(where("and", i), "combinational cycle through variable %d" % (ands[i, 0] >> 1))
                    if k >= 0 and state[k] == 0:
                        stack.append(k)
            else:
                stack.pop()
                if state[i] == 1:
                    state[i] = 2
                    order.append(i)
    return np.array(order, np.int64)


def _fold(M, ands):
    """Every variable's literal with constants folded, over ``ands`` in topological order: 0 / 1 for the constants,
    ``2 v + c`` for a variable v that stays a node (an input, a latch or an AND that does not fold)."""
    rl = 2 * np.arange(M + 1, dtype=np.int64)
    v, p, q = ands[:, 0] >> 1, ands[:, 1], ands[:, 2]
    direct = ((p >> 1) == 0) | ((q >> 1) == 0) | ((p >> 1) == (q >> 1))
    if not direct.any():                                      # nothing folds, so no literal changes
        return rl
    first = int(np.argmax(direct))                            # the ANDs before it keep their literals
    r = rl.tolist()
    for w, a, b in zip(v[first:].tolist(), p[first:].tolist(), q[first:].tolist()):
        x, y = r[a >> 1] ^ (a & 1), r[b >> 1] ^ (b & 1)
        if x > y:
            x, y = y, x
        if x == 0 or x ^ y == 1:                              # AND(0, y), AND(a, NOT a)
            r[w] = 0
        elif x == 1 or x == y:                                # AND(1, y), AND(a, a)
            r[w] = y
    return np.array(r, np.int64)


def read_aiger(path, kind="aig"):
    """One AIGER file (``.aag`` or ``.aig``, told apart by its header) as a circuit dict with ``x``, ``edge_index``,
    ``name``, ``lit`` and ``outputs``; the module docstring gives the node order, the folding, the latches and the
    literal encoding."""
    if kind not in CODE_TABLES:
        raise ValueError("kind must be one of %s, got %r" % (sorted(CODE_TABLES), kind))
    table = CODE_TABLES[kind]
    src = _Src(path)
    with open(path, "rb") as f:
        data = f.read()
    M, O, inputs, lat, outs, ands, where = _parse(src, data)
    pos = _check(src, M, inputs, lat, outs, ands, where)
    ands = ands[_topo_order(src, ands, pos, where)]
    rl = _fold(M, ands)
    ands = ands[rl[ands[:, 0] >> 1] == ands[:, 0]]           # the ANDs that stay nodes, in topological order
    fan = rl[ands[:, 1:] >> 1] ^ (ands[:, 1:] & 1)           # their fan-in literals after folding [A', 2]
    out = np.concatenate([outs[:O], lat[:, 1], outs[O:]])
    out = rl[out >> 1] ^ (out & 1)
    used = np.concatenate([fan.reshape(-1), out[out >= 2]])
    need_not = np.zeros(M + 1, bool)
    need_not[used[(used & 1) == 1] >> 1] = True
    in_var = np.concatenate([inputs, lat[:, 0]]) >> 1
    and_var = ands[:, 0] >> 1
    k = in_var.size
    node = np.full(M + 1, -1, np.int64)                       # node[0] = -1: the constant
    not_node = np.full(M + 1, -1, np.int64)
    node[in_var] = np.arange(k)
    in_not = in_var[need_not[in_var]]
    not_node[in_not] = k + np.arange(in_not.size)
    size = 1 + need_not[and_var].astype(np.int64)             # an AND and its NOT node, if any
    start = k + in_not.size + np.cumsum(size) - size
    node[and_var] = start
    not_node[and_var[size == 2]] = start[size == 2] + 1
    n = k + in_not.size + int(size.sum())
    gate = np.full(n, table.index("NOT"), np.int64)
    gate[:k] = table.index("INPUT")
    gate[start] = table.index("AND")
    has_not = np.flatnonzero(not_node >= 0)
    e_src = np.concatenate([node[has_not], np.where(fan & 1, not_node[fan >> 1], node[fan >> 1]).reshape(-1)])
    e_dst = np.concatenate([not_node[has_not], np.repeat(start, 2)])
    e = np.lexsort((e_src, e_dst))
    return {"x": np.stack([np.arange(n), gate], axis=1), "edge_index": np.stack([e_src[e], e_dst[e]], axis=1),
            "name": os.path.splitext(os.path.basename(str(path)))[0],
            "lit": 2 * node[rl >> 1] + (rl & 1), "outputs": 2 * node[out >> 1] + (out & 1)}


def read_aiger_files(paths, kind="aig"):
    """Circuit dicts of AIGER files: ``paths`` is a path or a list of them, each a file or a directory whose ``.aag`` /
    ``.aig`` files (not those of its subdirectories) are read in name order.  Circuits are named by file stem, which must
    be unique because ``write_npz`` stores circuits under their names."""
    files = []
    for p in [paths] if isinstance(paths, (str, os.PathLike)) else paths:
        if os.path.isdir(p):
            files += sorted(os.path.join(p, f) for f in os.listdir(p)
                            if f.endswith(SUFFIXES) and os.path.isfile(os.path.join(p, f)))
        else:
            files.append(p)
    circuits = [read_aiger(f, kind) for f in files]
    names = [c["name"] for c in circuits]
    for i, name in enumerate(names):
        if name in names[:i]:
            raise ValueError("%s: a circuit named %r was already read from %s" % (files[i], name, files[names.index(name)]))
    return circuits
