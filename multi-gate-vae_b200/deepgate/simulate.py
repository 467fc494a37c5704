"""Circuit labels by bit-parallel logic simulation on the GPU (csrc/logic_sim.cu): ``prob`` (probability that a node is 1
under random inputs) and the truth-table distance of node pairs (``tt_sim`` in a batch, ``tt_dis`` in ``labels.npz``).

    prob, tt_dis = simulate(G, "mig")                       # a CUDA batch, e.g. circuits_to_batch(circuits, "cuda")
    labelled = label_circuits(circuits, "mig", "cuda:0")    # synth-style circuit dicts -> copies with labels
    write_npz(labelled, "graphs.npz", "labels.npz", "mig")  # the reference's on-disk layouts, read back by NpzParser
    rep, complemented, n_split = equivalence_classes(G, "mig")   # functionally equal / complementary gates
    python -m deepgate.simulate --graphs graphs.npz --type mig --out DIR [--class-pairs K]
    python -m deepgate.simulate --aiger FILE_OR_DIR ... --type mig --out DIR  # AIGER netlists (deepgate/aiger.py)
    python -m deepgate.simulate --aiger FILE_OR_DIR ... --type xmg --map --out DIR  # mapped onto XMG gates first
    python -m deepgate.simulate --aiger FILE_OR_DIR ... --type mig --cycles 32 --warmup 8 --out DIR  # sequential

Gate functions by code: AIG {0 INPUT, 1 AND, 2 NOT}; MIG / XMG / XAG {0 INPUT, 1 MAJ, 2 NOT, 3 AND, 4 OR, 5 XOR}.  AND, OR
and XOR reduce over all their predecessors, NOT takes one, MAJ three.  Random mode: ``patterns`` (a multiple of 64) patterns;
word w of an INPUT is a splitmix64 hash of (seed, the INPUT's rank among the INPUTs of its own circuit, w), so a circuit's
labels do not depend on the batch it sits in or on how the words are split into passes.  Exhaustive mode: every input
assignment of the largest circuit (K inputs, K <= 24), ``max(64, 2^K)`` patterns: exact probabilities.  The counts are
integers, so results are deterministic.  There is no CPU path; ``oracle/logic_sim.py`` is the numpy reference of the tests.

Sequential mode (``cycles`` = C, csrc/logic_sim.cu's seq_sim_kernel), for netlists with latches (``read_aiger``'s
``latches``): ``patterns`` traces, each starting in the reset state -- a latch with reset 0 holds 0, with reset 1 holds 1,
an uninitialised one the random word its INPUT gets in random mode (trace word w).  In cycle t = 0 .. C-1 every primary
INPUT takes the random-mode word of global index t * T + w (T = patterns / 64), every node is evaluated from the primary
inputs and the state, and then every latch takes the value of its next-state literal.  ``ones`` and ``diff`` count the
cycles t in [warmup, C) only, a latch INPUT with the state it holds in cycle t, so ``prob`` and ``tt_dis`` are over
patterns * (C - warmup) samples.  A circuit without latches at warmup 0 gives exactly the combinational counts at
patterns * C patterns, and C = 1 with every latch uninitialised exactly those at ``patterns``.  The graph and the model
stay combinational: latch INPUTs are level-0 nodes.

Equivalence classes (csrc/sim_classes.cu): nodes of one circuit whose words are equal, or bitwise complementary, on every
simulated pattern -- exact functional equivalence in exhaustive mode, equality on the drawn patterns in random mode.

The package exports ``simulate``, ``simulate_counts``, ``equivalence_classes``, ``label_circuits`` and ``write_npz`` as
``deepgate.<name>``; the package
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
MAX_SEQ_WORDS = 2 ** 40                  # MGV_SEQ_MAX_WORDS: cycles x patterns / 64 input words, below the rank bits


def _is_int(v):
    return isinstance(v, (int, np.integer)) and not isinstance(v, bool)


def _fn_table(kind):
    if kind not in CODE_TABLES:
        raise ValueError("kind must be one of %s, got %r" % (sorted(CODE_TABLES), kind))
    names = CODE_TABLES[kind]
    return (ctypes.c_int32 * nat.NCODE)(*[_F[names[c]] if c < len(names) else _F["NONE"] for c in range(nat.NCODE)])


def _circuit_ids(G, n, device):
    """Circuit of every node (``G.batch`` / ``G.ptr``; neither = one circuit), int64 on ``device``."""
    batch = getattr(G, "batch", None)
    if batch is None or batch.numel() != n:
        ptr = getattr(G, "ptr", None)
        if ptr is not None and int(ptr[-1]) == n:
            batch = torch.repeat_interleave(torch.arange(ptr.numel() - 1, device=device), (ptr[1:] - ptr[:-1]).to(device))
        else:
            batch = torch.zeros(n, dtype=torch.long, device=device)
    return batch.to(device, torch.long)


def _input_ranks(G, code):
    """Rank of every INPUT among the INPUTs of its circuit (``G.batch`` / ``G.ptr``; neither = one circuit), and the
    largest INPUT count of any circuit.  Runs where the batch lives."""
    n = code.numel()
    batch = _circuit_ids(G, n, code.device)
    is_in = (code == 0).to(torch.long)
    per = torch.zeros(int(batch.max()) + 1 if n else 1, dtype=torch.long, device=code.device).index_add_(0, batch, is_in)
    base = torch.cumsum(per, 0) - per
    rank = torch.cumsum(is_in, 0) - 1 - base[batch]
    return rank.to(torch.int32).contiguous(), int(per.max()) if n else 0


class _Sim(object):
    """One simulation of a CUDA batch: argument checks at construction, then ``passes`` runs mgv_logic_sim_pass (or, with
    ``cycles``, mgv_seq_sim_pass) over every word of the patterns, ``W`` words at a time (the pass's buffers <=
    ``max_bytes``)."""

    def __init__(self, G, kind, patterns, seed, exhaustive, max_bytes, cycles=None, warmup=0, latches=None):
        self.table = _fn_table(kind)
        if not exhaustive and (int(patterns) <= 0 or int(patterns) % 64):
            raise ValueError("patterns must be a positive multiple of 64, got %r" % (patterns,))
        self.seq = cycles is not None
        if self.seq:
            if exhaustive:
                raise ValueError("exhaustive simulation does not take cycles: input sequences are drawn at random")
            if not _is_int(cycles) or not 1 <= cycles < 2 ** 31 or cycles * (int(patterns) // 64) > MAX_SEQ_WORDS:
                raise ValueError("cycles must be an integer >= 1 with cycles x patterns / 64 <= 2^40, got %r" % (cycles,))
            if not _is_int(warmup) or not 0 <= warmup < cycles:
                raise ValueError("warmup must be an integer in [0, cycles = %d), got %r" % (cycles, warmup))
            lat = torch.zeros(0, 3, dtype=torch.int64) if latches is None else torch.as_tensor(latches)
            if lat.dim() != 2 or lat.size(1) != 3:
                raise ValueError("latches must be int64 [L, 3] (node, next-state literal, reset), got shape %s"
                                 % (tuple(lat.shape),))
        elif warmup or latches is not None:
            raise ValueError("warmup and latches need cycles")
        self.rank, k = _input_ranks(G, G.gate.reshape(-1).to(torch.int32))
        if exhaustive and k > MAX_EXHAUSTIVE_INPUTS:
            raise ValueError("exhaustive simulation of a circuit with %d inputs (at most %d)" % (k, MAX_EXHAUSTIVE_INPUTS))
        if not G.edge_index.is_cuda:
            raise RuntimeError("mgv_b200: the batch must be on a CUDA device (no CPU path); call batch.to('cuda')")
        self.sch = schedule_for_batch(G)
        self.dev, self.n = self.sch.device, self.sch.N
        if self.seq:
            self.latches = lat.to(self.dev, torch.int64).contiguous()
            self.cycles, self.warmup = int(cycles), int(warmup)
            self.circuit = _circuit_ids(G, self.n, self.dev).to(torch.int32).contiguous()
        self.n_latch = self.latches.size(0) if self.seq else 0
        self.patterns = max(64, 1 << k) if exhaustive else int(patterns)
        self.samples = self.patterns * (self.cycles - self.warmup) if self.seq else self.patterns
        self.total = self.patterns // 64
        self.mode, self.seed = (1 if exhaustive else 0), int(seed) & (2 ** 64 - 1)
        self.max_bytes = max_bytes

    def words_per_pass(self):
        # per word: the nodes' words (and, with cycles, the latch states' words), plus the latch slot of every node
        per, fixed = (8 * (self.n + self.n_latch), 4 * self.n) if self.seq else (8 * self.n, 0)
        wmax = (int(self.max_bytes) - fixed) // per // SLICE_WORDS * SLICE_WORDS
        if wmax < 1:
            raise ValueError("max_bytes = %d is below one 32-byte slice per node (%d nodes)" % (self.max_bytes, self.n))
        return min(self.total, wmax)

    def sim_bytes(self, lib, W):
        return lib.mgv_seq_sim_bytes(self.n, self.n_latch, W) if self.seq else lib.mgv_logic_sim_bytes(self.n, W)

    def validate(self, lib, st, pairs, P):
        level = self.sch.level.reshape(-1).to(torch.int32).contiguous()
        ws = nat.workspace(max(16, 8 + 4 * self.n if self.seq else 0), self.dev)
        nat.check(lib.mgv_logic_sim_validate(self.sch.c_struct(), nat.ptr(self.sch.code), nat.ptr(level), self.table,
                                             nat.ptr(pairs), P, nat.ptr(ws), ws.numel(), st), "mgv_logic_sim_validate")
        if self.seq:
            nat.check(lib.mgv_seq_sim_validate(self.sch.c_struct(), nat.ptr(self.sch.code), self.table,
                                               nat.ptr(self.circuit), nat.ptr(self.latches), self.n_latch, self.cycles,
                                               self.warmup, nat.ptr(ws), ws.numel(), st), "mgv_seq_sim_validate")

    def passes(self, lib, st, W, sim, ones, pairs, P, diff):
        """Yields (first word, words) after each pass, with the pass's words in ``sim`` (without cycles)."""
        for first in range(0, self.total, W):
            w = min(W, self.total - first)
            if self.seq:
                nat.check(lib.mgv_seq_sim_pass(self.sch.c_struct(), nat.ptr(self.sch.code), nat.ptr(self.rank), self.table,
                                               nat.ptr(self.latches), self.n_latch, self.seed, first, w, self.total,
                                               self.cycles, self.warmup, nat.ptr(sim), sim.numel(), nat.ptr(ones),
                                               nat.ptr(pairs), P, nat.ptr(diff), st), "mgv_seq_sim_pass")
            else:
                nat.check(lib.mgv_logic_sim_pass(self.sch.c_struct(), nat.ptr(self.sch.code), nat.ptr(self.rank),
                                                 self.table, self.mode, self.seed, first, w, nat.ptr(sim),
                                                 nat.ptr(ones), nat.ptr(pairs), P, nat.ptr(diff), st), "mgv_logic_sim_pass")
            yield first, w


def simulate_counts(G, kind, patterns=32768, seed=0, exhaustive=False, max_bytes=2 ** 32, cycles=None, warmup=0,
                    latches=None):
    """Integer counts behind ``simulate``: (ones int64 [N], diff int64 [P], patterns) on the batch's device, ``ones[v]`` =
    patterns where node v is 1, ``diff[p]`` = patterns where the two nodes of ``G.tt_pair_index[:, p]`` differ.

    With ``cycles`` = C: sequential simulation of ``patterns`` traces from the reset state (module docstring); ``latches``
    int64 [L, 3] in batch-global node ids (INPUT node, next-state literal, reset 0 / 1 / 2 = uninitialised; None: no
    latches); the counts run over cycles [``warmup``, C), and the third value is samples = patterns * (C - warmup)."""
    s = _Sim(G, kind, patterns, seed, exhaustive, max_bytes, cycles, warmup, latches)
    dev, n = s.dev, s.n
    pairs = getattr(G, "tt_pair_index", None)
    pairs = (pairs if pairs is not None else torch.zeros(2, 0, dtype=torch.long, device=dev)).to(dev, torch.int64).contiguous()
    P = pairs.size(1)
    ones = torch.zeros(n, dtype=torch.int64, device=dev)
    diff = torch.zeros(P, dtype=torch.int64, device=dev)
    if n == 0:
        return ones, diff, s.samples
    W = s.words_per_pass()
    lib = nat.lib()
    st = nat.stream_of(dev)
    with nat.on_device(dev):
        s.validate(lib, st, pairs, P)
        sim = nat.workspace(s.sim_bytes(lib, W), dev)
        for _ in s.passes(lib, st, W, sim, ones, pairs, P, diff):
            pass
    return ones, diff, s.samples


def equivalence_classes(G, kind, patterns=32768, seed=0, exhaustive=False, max_bytes=2 ** 32):
    """Gates of a CUDA batch ``G`` grouped by the function they compute on the simulated patterns: (rep int64 [N],
    complemented bool [N], n_split int) on the batch's device.

    Two nodes of the same circuit share a class when their words are equal on every simulated pattern, or when one's are
    the bitwise NOT of the other's (then exactly one of them is ``complemented``).  In exhaustive mode that is exact
    functional equivalence; in random mode it is equality on the ``patterns`` random patterns, so nodes that differ only
    on patterns never drawn are grouped.  Nodes of different circuits are never grouped.  ``rep[v]`` is the batch-global
    id of the smallest node of v's class (a singleton is its own); ``complemented[v]`` is True when v computes the
    complement of ``rep[v]``.  Classes come from 64-bit hashes of every node's words (csrc/sim_classes.cu) and every
    member is then checked word by word against its representative; a member that fails becomes a singleton, and
    ``n_split`` counts them (expected 0).  Same arguments, checks and errors as ``simulate_counts``; the batch's
    ``tt_pair_index`` is not read.  When ``max_bytes`` forces several passes, the passes run twice (hash, then check)."""
    s = _Sim(G, kind, patterns, seed, exhaustive, max_bytes)
    dev, n = s.dev, s.n
    rep = torch.arange(n, dtype=torch.int64, device=dev)
    comp = torch.zeros(n, dtype=torch.uint8, device=dev)
    if n == 0:
        return rep, comp.bool(), 0
    W = s.words_per_pass()
    lib = nat.lib()
    st = nat.stream_of(dev)
    no_pairs = torch.zeros(2, 0, dtype=torch.int64, device=dev)
    circuit = _circuit_ids(G, n, dev).to(torch.int32).contiguous()
    with nat.on_device(dev):
        s.validate(lib, st, no_pairs, 0)
        sim = nat.workspace(lib.mgv_logic_sim_bytes(n, W), dev)
        ones = torch.zeros(n, dtype=torch.int64, device=dev)
        h = torch.zeros(2, n, dtype=torch.int64, device=dev)
        bit0 = torch.zeros(n, dtype=torch.uint8, device=dev)
        for first, w in s.passes(lib, st, W, sim, ones, no_pairs, 0, None):
            nat.check(lib.mgv_sim_signature_pass(nat.ptr(sim), n, w, first, nat.ptr(h[0]), nat.ptr(h[1]), nat.ptr(bit0), st),
                      "mgv_sim_signature_pass")
        ws = nat.workspace(lib.mgv_sim_classes_bytes(n), dev)
        nat.check(lib.mgv_sim_classes_group(nat.ptr(h[0]), nat.ptr(h[1]), nat.ptr(bit0), nat.ptr(circuit), n, nat.ptr(rep),
                                            nat.ptr(comp), nat.ptr(ws), ws.numel(), st), "mgv_sim_classes_group")
        bad = torch.zeros(n, dtype=torch.uint8, device=dev)

        def verify(w):
            nat.check(lib.mgv_sim_classes_verify_pass(nat.ptr(sim), n, w, nat.ptr(circuit), nat.ptr(rep), nat.ptr(comp),
                                                      nat.ptr(bad), st), "mgv_sim_classes_verify_pass")

        if W >= s.total:                                  # one pass: its words are still in sim
            verify(W)
        else:
            for _, w in s.passes(lib, st, W, sim, ones, no_pairs, 0, None):
                verify(w)
        n_split = ctypes.c_int64(0)
        nat.check(lib.mgv_sim_classes_split(n, nat.ptr(rep), nat.ptr(comp), nat.ptr(bad), nat.ptr(ws), ws.numel(),
                                            ctypes.byref(n_split), st), "mgv_sim_classes_split")
    return rep, comp.bool(), int(n_split.value)


def simulate(G, kind, patterns=32768, seed=0, exhaustive=False, max_bytes=2 ** 32, cycles=None, warmup=0, latches=None):
    """Signal probability and pair truth-table distance of a CUDA batch ``G``: (prob float32 [N, 1], tt_dis float32 [P]).
    ``kind`` picks the code table ("aig", "mig", "xmg", "xag"); ``max_bytes`` bounds the simulation buffer (N x words x
    8 bytes per pass; more passes when it is smaller).  A pass runs one CTA per 4 words, so a bound that leaves fewer than
    ~600 words per pass (148 SMs) idles most of the GPU: raise it for batches of millions of nodes (DESIGN.md §4.7).  Raises ``RuntimeError`` naming the first malformed node or pair.
    ``cycles``, ``warmup``, ``latches``: sequential simulation, as ``simulate_counts`` says; probabilities and distances
    are then over the counted (cycle, trace) samples, and a malformed latch raises ``RuntimeError`` naming it."""
    ones, diff, patterns = simulate_counts(G, kind, patterns, seed, exhaustive, max_bytes, cycles, warmup, latches)
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


def class_pair_count(rep):
    """Unordered node pairs inside the classes of ``rep`` (numpy int64 [N], each node's representative)."""
    m = np.bincount(np.asarray(rep, np.int64), minlength=len(rep)).astype(np.int64)
    return int((m * (m - 1) // 2).sum())


def _class_pairs_for(rep, index, k, seed):
    """Up to ``k`` distinct unordered pairs (smaller id first) drawn uniformly among the pairs inside the classes of
    ``rep`` (local ids of one circuit), with a generator seeded from ``seed`` and the circuit's index."""
    rep = np.asarray(rep, np.int64)
    members = np.argsort(rep, kind="stable")                 # nodes by class, ascending id within a class
    m = np.bincount(rep, minlength=len(rep)).astype(np.int64)
    cls = np.flatnonzero(m > 1)
    per = m[cls] * (m[cls] - 1) // 2
    total = int(per.sum())
    if total == 0 or k <= 0:
        return np.zeros((0, 2), dtype=np.int64)
    rng = np.random.default_rng([int(seed) & (2 ** 63 - 1), index, 1])
    t = np.sort(rng.choice(total, size=min(k, total), replace=False)).astype(np.int64)
    ends = np.cumsum(per)
    c = np.searchsorted(ends, t, side="right")               # class of each drawn pair
    u = t - (ends[c] - per[c])                              # pair index inside the class: (i, j), i < j, ordered by j
    j = ((1 + np.sqrt(1 + 8 * u.astype(np.float64))) / 2).astype(np.int64)
    j = np.where(j * (j - 1) // 2 > u, j - 1, j)
    j = np.where((j + 1) * j // 2 <= u, j + 1, j)
    i = u - j * (j - 1) // 2
    first = (np.cumsum(m) - m)[cls[c]]                       # where the class starts in `members`
    return np.stack([members[first + i], members[first + j]], axis=1).astype(np.int64)


def _draw_with_classes(G, chunk, i0, kind, n_pairs, class_pairs, seed, simulate_kw):
    """Pairs of the chunk's circuits without given pairs: class pairs, then random ones; sets ``G.tt_pair_index``."""
    rep = equivalence_classes(G, kind, **simulate_kw)[0].cpu().numpy()
    n0, glob = 0, []
    for j, c in enumerate(chunk):
        n = len(c["x"])
        if len(c["tt_pair_index"]) == 0:
            cp = _class_pairs_for(rep[n0:n0 + n] - n0, i0 + j, class_pairs, seed)
            c["tt_pair_index"] = np.concatenate([cp, _pairs_for(c, i0 + j, n_pairs - len(cp), seed)]).astype(np.int64)
            c["tt_sim"] = np.zeros(len(c["tt_pair_index"]), dtype=np.float32)
        glob.append(c["tt_pair_index"] + n0)
        n0 += n
    G.tt_pair_index = torch.from_numpy(np.concatenate(glob).T.copy()).to(G.edge_index.device)


def _batch_latches(chunk):
    """int64 [L, 3]: the ``latches`` of the chunk's circuit dicts in batch-global node ids."""
    rows, n0 = [], 0
    for c in chunk:
        lat = np.asarray(c.get("latches", np.zeros((0, 3))), np.int64).reshape(-1, 3).copy()
        lat[:, 0] += n0
        lat[:, 1] += np.where(lat[:, 1] >= 0, 2 * n0, 0)
        rows.append(lat)
        n0 += len(c["x"])
    return torch.from_numpy(np.concatenate(rows) if rows else np.zeros((0, 3), np.int64))


def label_circuits(circuits, kind, device, batch_size=64, n_pairs=64, class_pairs=0, **simulate_kw):
    """Copies of synth-style circuit dicts (``x`` with the gate code in column 1, ``edge_index`` [E, 2]) with ``prob`` [N],
    ``tt_pair_index`` [P, 2] and ``tt_sim`` [P] (the truth-table DISTANCE, what the func loss consumes) filled in.  A circuit's
    non-empty ``tt_pair_index`` is kept; otherwise ``n_pairs`` pairs of distinct nodes are drawn with a generator seeded from
    ``seed`` and the circuit's index.  Circuits are simulated ``batch_size`` at a time on ``device``.

    ``class_pairs = K > 0``: the pairs of a circuit without given pairs start with up to K pairs drawn uniformly among the
    pairs inside its classes of ``equivalence_classes`` (distance exactly 0, or exactly 1 for a complemented pair), and
    ``n_pairs`` minus those are drawn at random as above.  Those pairs are labelled by the same simulation as the others.
    ``class_pairs = 0`` gives the same output as before the option existed.

    ``cycles = C`` (and ``warmup``, as for ``simulate_counts``): sequential labels, from each dict's ``latches`` (as
    ``read_aiger`` and ``map_circuits`` give them; a dict without is combinational).  Equivalence classes are a
    combinational notion, so ``class_pairs`` must then be 0."""
    if isinstance(class_pairs, bool) or not isinstance(class_pairs, (int, np.integer)) or class_pairs < 0:
        raise ValueError("class_pairs must be an integer >= 0, got %r" % (class_pairs,))
    if class_pairs > n_pairs:
        raise ValueError("class_pairs = %d exceeds n_pairs = %d" % (class_pairs, n_pairs))
    simulate_kw = dict(simulate_kw)
    seq = simulate_kw.get("cycles") is not None
    if seq and class_pairs > 0:
        raise ValueError("class_pairs needs combinational simulation: it does not take cycles")
    if "latches" in simulate_kw:
        raise ValueError("label_circuits takes the latches from each circuit dict's 'latches'")
    from .parser_func_others import circuits_to_batch
    seed = simulate_kw.get("seed", 0)
    out = []
    for i0 in range(0, len(circuits), batch_size):
        chunk = []
        for j, c in enumerate(circuits[i0:i0 + batch_size]):
            c = dict(c)
            # with class pairs, a circuit without given pairs gets its pairs once its classes are known
            c["tt_pair_index"] = _pairs_for(c, i0 + j, 0 if class_pairs else n_pairs, seed)
            c["prob"] = np.zeros(len(c["x"]), dtype=np.float32)
            c["tt_sim"] = np.zeros(len(c["tt_pair_index"]), dtype=np.float32)
            chunk.append(c)
        G = circuits_to_batch(chunk, device)
        if class_pairs > 0:
            _draw_with_classes(G, chunk, i0, kind, n_pairs, class_pairs, seed, simulate_kw)
        if seq:
            simulate_kw["latches"] = _batch_latches(chunk)
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
                                 description="Label the circuits of a graphs.npz or of AIGER files by logic simulation on "
                                             "cuda:0 and write DIR/graphs.npz (+ DIR/labels.npz for mig / xmg / xag), "
                                             "readable by NpzParser.")
    src = ap.add_mutually_exclusive_group(required=True)
    src.add_argument("--graphs", help="input graphs.npz (the reference layout of --type)")
    src.add_argument("--aiger", nargs="+", metavar="FILE_OR_DIR",
                     help="input AIGER netlists: .aag / .aig files, or directories of them (deepgate/aiger.py)")
    ap.add_argument("--type", required=True, choices=sorted(CODE_TABLES))
    ap.add_argument("--out", required=True, help="output directory")
    ap.add_argument("--patterns", type=int, default=32768, help="random patterns, a multiple of 64")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--exhaustive", action="store_true", help="all input assignments (circuits of at most 24 inputs)")
    ap.add_argument("--pairs", type=int, default=64, help="node pairs drawn per circuit that has none")
    ap.add_argument("--class-pairs", type=int, default=0,
                    help="of those, up to this many drawn among functionally equivalent or complementary nodes")
    ap.add_argument("--map", action="store_true",
                    help="with --aiger and --type mig / xmg / xag: read the files as AIGs and map them onto the gates of "
                         "--type on cuda:0 first (deepgate/mapping.py)")
    ap.add_argument("--cycles", type=int, default=None,
                    help="with --aiger: simulate this many clock cycles from the latches' reset state; the labels "
                         "count every (cycle, trace) from --warmup on")
    ap.add_argument("--warmup", type=int, default=0, help="with --cycles: cycles simulated before counting starts")
    args = ap.parse_args(argv)
    if not 0 <= args.class_pairs <= args.pairs:
        ap.error("--class-pairs must be in [0, --pairs]")
    if args.cycles is None and args.warmup:
        ap.error("--warmup takes --cycles")
    if args.cycles is not None:
        if not args.aiger:
            ap.error("--cycles takes --aiger input (the --graphs layout has no latches)")
        if args.exhaustive or args.class_pairs:
            ap.error("--cycles does not combine with --exhaustive or --class-pairs")
        if args.cycles < 1 or not 0 <= args.warmup < args.cycles:
            ap.error("--cycles must be >= 1 and --warmup in [0, --cycles)")
    if args.map and (args.graphs or args.type == "aig"):
        ap.error("--map takes --aiger input and --type mig, xmg or xag")
    if args.aiger:
        from .aiger import read_aiger_files
        circuits = read_aiger_files(args.aiger, "aig" if args.map else args.type)
        dropped = sum(int((c["outputs"] < 0).sum()) for c in circuits)
        if dropped:
            print("dropped %d outputs that fold to constants" % dropped)
        if args.map:
            from .mapping import gate_counts, map_circuits
            ands = sum(int((c["x"][:, 1] == 1).sum()) for c in circuits)
            circuits = map_circuits(circuits, args.type, "cuda:0")
            counts = gate_counts(circuits, args.type)
            print("mapped %d circuits: %d ANDs in; out %s" % (len(circuits), ands, ", ".join(
                "%d %s" % (counts[g], g) for g in CODE_TABLES[args.type] if g != "INPUT")))
    else:
        circuits = read_circuits(args.graphs, args.type)
    seq = {}
    if args.cycles is not None:
        seq = {"cycles": args.cycles, "warmup": args.warmup}
        print("simulating %d latches over %d cycles (%d counted)"
              % (sum(len(c["latches"]) for c in circuits), args.cycles, args.cycles - args.warmup))
    labelled = label_circuits(circuits, args.type, "cuda:0", n_pairs=args.pairs, class_pairs=args.class_pairs,
                              patterns=args.patterns, seed=args.seed, exhaustive=args.exhaustive, **seq)
    os.makedirs(args.out, exist_ok=True)
    gp, lp = write_npz(labelled, os.path.join(args.out, "graphs.npz"), os.path.join(args.out, "labels.npz"), args.type)
    print("labelled %d circuits -> %s%s" % (len(labelled), gp, "" if lp == gp else ", " + lp))


if __name__ == "__main__":
    main()
