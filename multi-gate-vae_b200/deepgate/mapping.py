"""Map AIGs onto the gates of a MIG, XMG or XAG on the GPU (csrc/map_cuts.cu): 3-input cut enumeration with truth tables,
single-gate matching and an area-flow cover, so that AIGER netlists become circuits of the gate types those models have.

    mapped = map_circuits(read_aiger_files(paths, "aig"), "xmg", "cuda:0")
    python -m deepgate.simulate --aiger FILE_OR_DIR ... --type xmg --map --out DIR

Input: AIG-coded circuit dicts (INPUT 0, AND 1, NOT 2; ``read_aiger(path, "aig")``, ``synth.make_circuit("aig", ...)``),
ANDs of fan-in 2, NOTs of fan-in 1, every edge from a lower to a higher node id.
Gate library (AND, OR and XOR reduce over all their inputs, as the simulator defines them):
  * ``mig``: AND2, OR2, MAJ3;  ``xag``: AND2, XOR2 (an OR is an AND with complemented inputs and output);
  * ``xmg``: AND2, OR2, XOR2, XOR3, MAJ3.
Every gate input and the output may be complemented; complements become NOT nodes.  ``MATCH[kind]`` maps each 8-bit
truth table (leaf i is variable i) to one gate, input-complement mask and output complement -- the realisation with the
fewest complements, then the first gate in the order above -- or to -1.
Cuts (the kernel's header comment has the exact definitions): a cut is at most 3 leaves, non-NOT nodes; every AND node's
cuts are the unions of its fan-ins' cut sets, support reduced, without duplicates or dominated cuts, ranked by area flow
in integer fixed point and cut to ``CUTS_KEPT``; a node with a cut of at most one leaf is a constant or an alias of
another node's literal.  A node's best cut is its best-ranked cut that matches a gate.  The cover marks the nodes of the
outputs (of the fan-out-free nodes, for a dict without ``outputs``) and, from the last level down, the leaves of every
marked node's best cut.  Each marked AND that is not an alias becomes one gate.
Output dict, in the layout and codes of ``kind``: ``x``, ``edge_index`` [E, 2] sorted by (dst, src), ``name``,
``outputs`` (each output literal over the new nodes, ``2 node + complemented``; -2 / -1 the constants), ``origin``
int64 [N']: the literal over the input circuit's nodes that each new node computes, and, when the input has them,
``latches`` [L, 3] with the latch INPUT nodes and next-state literals over the new nodes (resets as given).  Node
order: the INPUTs in their order (an AIG whose INPUTs come first, as ``read_aiger`` gives, keeps their ids), their NOT
nodes, then the gates by the id of the AND they replace, each directly followed by its NOT node if it has one; one NOT
node per complemented node, shared by all of its uses.  Labels of the input are not carried over.
"""
import ctypes

import numpy as np
import torch

from . import _native as nat
from .schedule import schedule_for_batch
from .simulate import CODE_TABLES

CUTS_KEPT = 16                                               # MAP_C of csrc/map_cuts.cu
NO_ALIAS = -3                                                # alias entry of a node that is not an alias
GATES = ("AND2", "OR2", "XOR2", "XOR3", "MAJ3")
_ARITY = {"AND2": 2, "OR2": 2, "XOR2": 2, "XOR3": 3, "MAJ3": 3}
_CODE_NAME = {"AND2": "AND", "OR2": "OR", "XOR2": "XOR", "XOR3": "XOR", "MAJ3": "MAJ"}
LIBRARY = {"mig": ("AND2", "OR2", "MAJ3"), "xag": ("AND2", "XOR2"), "xmg": ("AND2", "OR2", "XOR2", "XOR3", "MAJ3")}
_AIG_INPUT, _AIG_AND, _AIG_NOT = 0, 1, 2
_VAR = (0xAA, 0xCC, 0xF0)                                    # truth tables of variables 0, 1, 2


def _gate_table(gate, mask, out):
    v = [_VAR[i] ^ (0xFF if mask >> i & 1 else 0) for i in range(_ARITY[gate])]
    if gate == "AND2":
        t = v[0] & v[1]
    elif gate == "OR2":
        t = v[0] | v[1]
    elif gate in ("XOR2", "XOR3"):
        t = v[0] ^ v[1] ^ (v[2] if gate == "XOR3" else 0)
    else:
        t = (v[0] & v[1]) | (v[0] & v[2]) | (v[1] & v[2])
    return t ^ (0xFF if out else 0)


def _match_table(kind):
    """int32 [256]: gate index in ``GATES`` | input-complement mask << 3 | output complement << 6, or -1."""
    table = np.full(256, -1, np.int32)
    rank = {}
    for lib_pos, gate in enumerate(LIBRARY[kind]):
        for mask in range(1 << _ARITY[gate]):
            for out in (0, 1):
                t = _gate_table(gate, mask, out)
                key = (bin(mask).count("1") + out, lib_pos)
                if t not in rank or key < rank[t]:
                    rank[t] = key
                    table[t] = GATES.index(gate) | mask << 3 | out << 6
    return table


MATCH = {kind: _match_table(kind) for kind in LIBRARY}


def decode_match(entry):
    """(gate name, input-complement mask, output complement) of a ``MATCH`` entry >= 0."""
    return GATES[entry & 7], (entry >> 3) & 7, (entry >> 6) & 1


def _name(c, i):
    return c.get("name") or "circuit %d" % i


def _check(c, i):
    """ValueError naming the circuit and the node or edge when ``c`` is not an AIG the mapper takes."""
    code = np.asarray(c["x"])[:, 1].astype(np.int64)
    n = len(code)
    ei = np.asarray(c["edge_index"], np.int64).reshape(-1, 2)
    bad = np.flatnonzero(~np.isin(code, (_AIG_INPUT, _AIG_AND, _AIG_NOT)))
    if bad.size:
        raise ValueError("%s: node %d has gate code %d; the mapper takes AIGs (INPUT 0, AND 1, NOT 2)"
                         % (_name(c, i), bad[0], code[bad[0]]))
    bad = np.flatnonzero((ei[:, 0] < 0) | (ei[:, 1] >= n) | (ei[:, 0] >= ei[:, 1]))
    if bad.size:
        e = int(bad[0])
        raise ValueError("%s: edge %d (%d -> %d): every edge must go from a lower to a higher node id in [0, %d)"
                         % (_name(c, i), e, ei[e, 0], ei[e, 1], n))
    deg = np.bincount(ei[:, 1], minlength=n)
    want = np.array([0, 2, 1])[code]
    bad = np.flatnonzero(deg != want)
    if bad.size:
        v = int(bad[0])
        raise ValueError("%s: node %d (%s) has fan-in %d, needs %d"
                         % (_name(c, i), v, ("INPUT", "AND", "NOT")[code[v]], deg[v], want[v]))


def _roots(c):
    """Root nodes of the cover: the nodes of the output literals, or the fan-out-free nodes of a dict without outputs."""
    if "outputs" in c:
        out = np.asarray(c["outputs"], np.int64)
        return out[out >= 0] >> 1
    n = len(c["x"])
    return np.flatnonzero(np.bincount(np.asarray(c["edge_index"], np.int64).reshape(-1, 2)[:, 0], minlength=n) == 0)


def _and_levels(sch):
    """int32 [n, 2] (first position in ``order``, count) of the AND nodes of each level that has some, in level order."""
    seg = sch.seg_ptr.cpu().numpy().astype(np.int64).reshape(-1)
    lv = np.arange(sch.L) * nat.NCODE
    beg, end = seg[lv + _AIG_AND], seg[lv + _AIG_AND + 1]
    keep = end > beg
    return np.ascontiguousarray(np.stack([beg[keep], (end - beg)[keep]], axis=1).astype(np.int32))


class _Batch(object):
    """One batch of checked circuits on ``device``: the level schedule and buffers at construction, ``run`` launches the
    enumeration and the cover (asynchronous), ``arrays`` copies the per-node arrays back."""

    def __init__(self, circuits, kind, device):
        from .parser_func_others import circuits_to_batch
        self.dev = dev = torch.device(device)
        chunk = [{"x": c["x"], "edge_index": c["edge_index"], "prob": np.zeros(len(c["x"]), np.float32),
                  "tt_sim": np.zeros(0, np.float32), "tt_pair_index": np.zeros((0, 2), np.int64)} for c in circuits]
        G = circuits_to_batch(chunk, dev)
        self.sch = schedule_for_batch(G, streams=1)
        n = max(self.sch.N, 1)
        self.sizes = [len(c["x"]) for c in circuits]
        self.starts = np.concatenate([[0], np.cumsum(self.sizes)]).astype(np.int64)
        self.levels = _and_levels(self.sch)
        self.roots = torch.from_numpy(np.concatenate([_roots(c) + s for c, s in zip(circuits, self.starts)])
                                      .astype(np.int32)).to(dev)
        self.best = torch.empty(n, 4, dtype=torch.int32, device=dev)
        self.match = torch.empty(n, dtype=torch.int32, device=dev)
        self.flow = torch.empty(n, dtype=torch.int32, device=dev)
        self.alias = torch.empty(n, dtype=torch.int32, device=dev)
        self.required = torch.empty(n, dtype=torch.uint8, device=dev)
        self.table = torch.from_numpy(MATCH[kind]).to(dev)
        self.ws = nat.workspace(nat.lib().mgv_map_cuts_bytes(self.sch.N), dev)

    def run(self):
        lib, sch = nat.lib(), self.sch
        lv = ctypes.c_void_p(self.levels.ctypes.data)
        st = nat.stream_of(self.dev)
        with nat.on_device(self.dev):
            nat.check(lib.mgv_map_cuts(sch.c_struct(), nat.ptr(sch.code), nat.ptr(self.table), lv, len(self.levels),
                                       nat.ptr(self.best), nat.ptr(self.match), nat.ptr(self.flow), nat.ptr(self.alias),
                                       nat.ptr(self.ws), self.ws.numel(), st), "mgv_map_cuts")
            nat.check(lib.mgv_map_cover(sch.c_struct(), nat.ptr(sch.code), nat.ptr(self.roots), self.roots.numel(), lv,
                                        len(self.levels), nat.ptr(self.best), nat.ptr(self.alias),
                                        nat.ptr(self.required), st), "mgv_map_cover")

    def arrays(self):
        best, match = self.best.cpu().numpy(), self.match.cpu().numpy()
        flow = self.flow.cpu().numpy().view(np.uint32).astype(np.int64)
        alias, required = self.alias.cpu().numpy(), self.required.cpu().numpy().astype(bool)
        out = []
        for s, size in zip(self.starts[:-1], self.sizes):
            b = best[s:s + size].copy()
            b[:, :3] = np.where(b[:, :3] >= 0, b[:, :3] - s, -1)
            a = alias[s:s + size]
            out.append({"required": required[s:s + size].copy(), "best": b, "match": match[s:s + size].copy(),
                        "flow": flow[s:s + size].copy(), "alias": np.where(a >= 0, a - 2 * s, a).astype(np.int32)})
        return out


def _node_arrays(circuits, kind, device):
    """The per-node arrays the mapped circuits are emitted from, for one batch of checked circuits on ``device``: one dict
    per circuit, in its local node ids, with ``required`` bool [n], ``best`` int32 [n, 4] (best cut leaves, -1 padded;
    table | leaves << 8), ``match`` int32 [n] (``MATCH`` entry of the best cut), ``flow`` int64 [n] and ``alias`` int32 [n]
    (a literal, -2 / -1 the constants, ``NO_ALIAS``).  INPUTs and aliases have match -1 and flow 0; an alias's best cut is
    its alias cut."""
    b = _Batch(circuits, kind, device)
    b.run()
    return b.arrays()


def _resolve_nots(code, ei):
    """int64 [n]: every node's literal ``2 u + c`` over the non-NOT node u at the end of its NOT chain."""
    n = len(code)
    pred = np.arange(n)
    nots = code == _AIG_NOT
    pred[ei[nots[ei[:, 1]], 1]] = ei[nots[ei[:, 1]], 0]
    flip = nots.astype(np.int64)
    while True:                                              # pointer jumping: log(chain length) rounds
        nxt = pred[pred]
        if np.array_equal(nxt, pred):
            break
        flip = flip ^ flip[pred]
        pred = nxt
    return 2 * pred + flip


def emit(c, kind, arrays):
    """The mapped circuit dict of AIG ``c`` (module docstring) from its per-node arrays (``_node_arrays``)."""
    table = CODE_TABLES[kind]
    code = np.asarray(c["x"])[:, 1].astype(np.int64)
    ei = np.asarray(c["edge_index"], np.int64).reshape(-1, 2)
    alias = arrays["alias"].astype(np.int64)
    res = _resolve_nots(code, ei)

    def final(lit):                                          # literal over the input -> over non-NOT, non-alias nodes
        lit = np.asarray(lit, np.int64)
        const = lit < 0
        r = res[np.where(const, 0, lit >> 1)] ^ (lit & 1)
        a = alias[r >> 1]
        return np.where(const, lit, np.where(a != NO_ALIAS, a ^ (r & 1), r))

    inputs = np.flatnonzero(code == _AIG_INPUT)
    gates = np.flatnonzero(arrays["required"] & (code == _AIG_AND) & (alias == NO_ALIAS))
    m = arrays["match"][gates].astype(np.int64)
    if (m < 0).any():
        raise RuntimeError("mgv_b200 map: required node %d has no matched cut" % gates[np.argmax(m < 0)])
    gate_idx, mask, oc = m & 7, (m >> 3) & 7, (m >> 6) & 1
    k = (arrays["best"][gates, 3].astype(np.int64) >> 8) & 3
    leaves = arrays["best"][gates, :3].astype(np.int64)
    n = len(code)
    out_c = np.zeros(n, np.int64)                            # output complement of the gate replacing each AND
    out_c[gates] = oc
    slot = np.arange(3)[None, :] < k[:, None]
    use_node, use_dst = leaves[slot], np.repeat(gates, k)
    use_comp = ((mask[:, None] >> np.arange(3)[None, :]) & 1)[slot] ^ out_c[use_node]
    roots = np.asarray(c["outputs"], np.int64) if "outputs" in c else 2 * _roots(c)
    rl = final(roots)
    o_node = rl[rl >= 0] >> 1
    o_comp = (rl[rl >= 0] & 1) ^ out_c[o_node]
    need_not = np.zeros(n, bool)
    need_not[use_node[use_comp == 1]] = True
    need_not[o_node[o_comp == 1]] = True
    node, not_node = np.full(n, -1, np.int64), np.full(n, -1, np.int64)
    node[inputs] = np.arange(inputs.size)
    in_not = inputs[need_not[inputs]]
    not_node[in_not] = inputs.size + np.arange(in_not.size)
    size = 1 + need_not[gates].astype(np.int64)
    start = inputs.size + in_not.size + np.cumsum(size) - size
    node[gates] = start
    not_node[gates[size == 2]] = start[size == 2] + 1
    total = inputs.size + in_not.size + int(size.sum())
    gcode = np.full(total, table.index("NOT"), np.int64)
    gcode[:inputs.size] = table.index("INPUT")
    gcode[start] = np.array([table.index(_CODE_NAME[g]) for g in GATES], np.int64)[gate_idx]
    origin = np.empty(total, np.int64)
    origin[:inputs.size] = 2 * inputs
    origin[not_node[in_not]] = 2 * in_not + 1
    origin[start] = 2 * gates + oc
    has = size == 2
    origin[start[has] + 1] = 2 * gates[has] + (1 - oc[has])
    has_not = np.flatnonzero(not_node >= 0)
    e_src = np.concatenate([node[has_not], np.where(use_comp == 1, not_node[use_node], node[use_node])])
    e_dst = np.concatenate([not_node[has_not], node[use_dst]])
    e = np.lexsort((e_src, e_dst))

    def new_lit(rl):                                         # final literal -> literal over the new nodes
        u = np.maximum(rl, 0) >> 1
        return np.where(rl >= 0, 2 * node[u] + ((rl & 1) ^ out_c[u]), rl).astype(np.int64)

    out = {"x": np.stack([np.arange(total), gcode], axis=1), "edge_index": np.stack([e_src[e], e_dst[e]], axis=1),
           "name": c.get("name", ""), "outputs": new_lit(rl), "origin": origin}
    if "latches" in c:                                       # next states are outputs too, so their nodes exist
        lat = np.asarray(c["latches"], np.int64).reshape(-1, 3)
        out["latches"] = np.stack([node[lat[:, 0]], new_lit(final(lat[:, 1])), lat[:, 2]], axis=1).reshape(-1, 3)
    return out


def map_circuits(circuits, kind, device, batch_size=64):
    """Mapped copies of AIG circuit dicts onto the gates of ``kind`` ("mig", "xmg" or "xag"), ``batch_size`` circuits at
    a time on the CUDA ``device``; see the module docstring for the library, the definitions and the output."""
    if kind not in LIBRARY:
        raise ValueError("kind must be one of %s (the input is an AIG), got %r" % (sorted(LIBRARY), kind))
    dev = torch.device(device)
    if dev.type != "cuda":
        raise ValueError("map_circuits runs on a CUDA device (no CPU path), got %s" % dev)
    for i, c in enumerate(circuits):
        _check(c, i)
    out = []
    for i0 in range(0, len(circuits), batch_size):
        chunk = circuits[i0:i0 + batch_size]
        for c, arrays in zip(chunk, _node_arrays(chunk, kind, dev)):
            out.append(emit(c, kind, arrays))
    return out


def gate_counts(circuits, kind):
    """{code name: number of nodes} over the circuits of ``kind`` (the CLI's summary)."""
    names = CODE_TABLES[kind]
    counts = np.bincount(np.concatenate([np.asarray(c["x"])[:, 1] for c in circuits]).astype(np.int64),
                         minlength=len(names)) if circuits else np.zeros(len(names), np.int64)
    return {names[i]: int(counts[i]) for i in range(len(names))}
