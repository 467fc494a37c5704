"""Per-node Python reference of deepgate.map_circuits's enumeration, ranking and cover (csrc/map_cuts.cu), the oracle of
tests/test_map.py.  Same definitions as the kernel's header comment; it reuses ``MATCH`` and ``emit`` from
deepgate/mapping.py.  Plain: one node at a time in id order (a topological order), for circuits of a few thousand nodes."""
import numpy as np

from deepgate import mapping as MP

C = MP.CUTS_KEPT
UNIT = 256
NEG = (0x55, 0x33, 0x0F)


def _expand(tt, leaves, u):
    pos = [u.index(l) for l in leaves]
    out = 0
    for m in range(8):
        idx = 0
        for i, p in enumerate(pos):
            idx |= ((m >> p) & 1) << i
        out |= ((tt >> idx) & 1) << m
    return out


def _reduce(leaves, tt):
    keep = [i for i in range(len(leaves)) if ((tt >> (1 << i)) ^ tt) & NEG[i]]
    if len(keep) == len(leaves):
        return leaves, tt
    out = 0
    for m in range(8):
        idx = 0
        for j, i in enumerate(keep):
            idx |= ((m >> j) & 1) << i
        out |= ((tt >> idx) & 1) << m
    return tuple(leaves[i] for i in keep), out


def node_arrays(c, kind):
    """The dict of ``mapping._node_arrays`` for one circuit: required, best, match, flow, alias (local ids)."""
    match = MP.MATCH[kind]
    code = np.asarray(c["x"])[:, 1].astype(np.int64)
    ei = np.asarray(c["edge_index"], np.int64).reshape(-1, 2)
    n = len(code)
    preds = [[] for _ in range(n)]
    for s, d in ei.tolist():
        preds[d].append(s)
    res = MP._resolve_nots(code, ei).tolist()
    fanout = [0] * n
    for v in range(n):
        if code[v] == 1:
            for s in preds[v]:
                fanout[res[s] >> 1] += 1
    cuts = [[] for _ in range(n)]                            # kept cuts: (leaves tuple, table)
    flow = [0] * n
    alias = [MP.NO_ALIAS] * n
    best = np.full((n, 4), -1, np.int32)
    best[:, 3] = 0
    bmatch = np.full(n, -1, np.int32)

    def cflow(leaves, tt):
        f = UNIT if match[tt] >= 0 else 2 * UNIT
        for u in leaves:
            f += flow[u] // max(1, fanout[u])
        return min(f, 0xFFFFFFFF)

    def key(leaves, tt):
        return (cflow(leaves, tt), len(leaves), leaves)

    def offered(u):
        if alias[u] != MP.NO_ALIAS:
            return [cuts[u][0]]
        return [((u,), 0xAA)] + cuts[u]

    for v in range(n):
        if code[v] != 1:
            continue
        f0, f1 = sorted(res[s] for s in preds[v])
        c0, c1 = (0xFF if f0 & 1 else 0), (0xFF if f1 & 1 else 0)
        cand = []
        for x in offered(f0 >> 1):
            for y in offered(f1 >> 1):
                u = tuple(sorted(set(x[0]) | set(y[0])))
                if len(u) > 3:
                    continue
                tt = (_expand(x[1], x[0], u) ^ c0) & (_expand(y[1], y[0], u) ^ c1) & 0xFF
                w = _reduce(u, tt)
                sw = set(w[0])
                if any(set(q[0]) <= sw for q in cand):
                    continue
                cand = [q for q in cand if not sw <= set(q[0])] + [w]
        small = [q for q in cand if len(q[0]) <= 1]
        if small:
            a = min(small, key=lambda q: key(*q))
            cuts[v] = [a]
            best[v, :len(a[0])] = a[0]
            best[v, 3] = a[1] | len(a[0]) << 8
            alias[v] = (-1 if a[1] else -2) if not a[0] else 2 * a[0][0] + (a[1] == 0x55)
            continue
        ranked = sorted(cand, key=lambda q: key(*q))
        kept = ranked[:C]
        if cand[0] not in kept:
            kept[-1] = cand[0]
        cuts[v] = kept
        b = min((q for q in cand if match[q[1]] >= 0), key=lambda q: key(*q))
        best[v, :len(b[0])] = b[0]
        best[v, 3] = b[1] | len(b[0]) << 8
        bmatch[v] = match[b[1]]
        flow[v] = cflow(*b)
    required = np.zeros(n, bool)
    for r in MP._roots(c).tolist():
        u = res[r] >> 1
        if alias[u] != MP.NO_ALIAS:
            if alias[u] < 0:
                continue
            u = alias[u] >> 1
        required[u] = True
    for v in range(n - 1, -1, -1):                           # reverse id order: every leaf has a smaller id
        if required[v] and code[v] == 1 and alias[v] == MP.NO_ALIAS:
            k = best[v, 3] >> 8
            required[best[v, :k]] = True
    return {"required": required, "best": best, "match": bmatch, "flow": np.array(flow, np.int64),
            "alias": np.array(alias, np.int32)}


def map_circuit(c, kind):
    """The mapped circuit dict, as ``map_circuits`` gives it, from the reference's per-node arrays."""
    return MP.emit(c, kind, node_arrays(c, kind))
