"""Functional equivalence classes from simulation words (deepgate.equivalence_classes, csrc/sim_classes.cu) against
the numpy reference tests/sim_classes_oracle.py, and label pairs drawn from the classes (label_circuits(class_pairs=K)).
CPU: the oracle on constructed equivalences in every code table, pass independence, the class-pair draw, argument errors.
GPU: partitions and polarity bit-equal to the oracle over gate mixes, modes, depths, pass splits and batch placement;
the verification entry point on wrong assignments; class pairs labelled 0 / 1 through to one training epoch."""
import ctypes
import os

import numpy as np
import pytest
import torch

from sim_classes_oracle import classes as oracle_classes_of


def circuit(codes, edges, n_pi):
    """A hand-built circuit dict: ``n_pi`` INPUTs, then gates with ``codes``; ``edges`` (src, dst) pairs."""
    code = np.array([0] * n_pi + list(codes), dtype=np.int64)
    x = np.stack([np.arange(code.size), code], axis=1)
    ei = np.array(edges, dtype=np.int64).reshape(-1, 2)
    return {"x": x, "edge_index": ei, "prob": np.zeros(code.size, np.float32),
            "tt_pair_index": np.zeros((0, 2), np.int64), "tt_sim": np.zeros(0, np.float32)}


def partition(rep, comp):
    """Classes as a set of (representative, member ids, member polarities)."""
    rep, comp = np.asarray(rep, np.int64), np.asarray(comp, bool)
    out = set()
    for r in np.unique(rep):
        m = np.flatnonzero(rep == r)
        out.add((int(r), tuple(int(v) for v in m), tuple(bool(b) for b in comp[m])))
    return out


def expected_partition(n, classes):
    """rep / complemented of ``n`` nodes from ``classes``: lists of (node, complemented) with the smallest node first."""
    rep, comp = np.arange(n), np.zeros(n, bool)
    for cls in classes:
        r = min(v for v, _ in cls)
        for v, c in cls:
            rep[v], comp[v] = r, c
    return partition(rep, comp)


# MIG / XMG / XAG codes: 0 INPUT, 1 MAJ, 2 NOT, 3 AND, 4 OR, 5 XOR; AIG: 0 INPUT, 1 AND, 2 NOT.
# (kinds, gate codes after the inputs, edges, inputs, classes of more than one node as [(node, complemented)])
CONSTRUCTED = {
    "duplicate": (["aig"], [1, 1, 2, 2, 1],                     # 3 = 4 = AND(a, b); 5, 6 their NOTs; 7 = AND(a, c)
                  [(0, 3), (1, 3), (0, 4), (1, 4), (3, 5), (4, 6), (0, 7), (2, 7)], 3,
                  [[(3, False), (4, False), (5, True), (6, True)]]),
    "double_negation": (["aig", "mig", "xmg", "xag"], [2, 2, 2],      # 3 = NOT a, 4 = NOT 3 (= a); 5 = NOT b
                        [(0, 3), (3, 4), (1, 5)], 3,
                        [[(0, False), (3, True), (4, False)], [(1, False), (5, True)]]),
    "de_morgan": (["mig", "xmg", "xag"], [3, 2, 2, 2, 4, 4],   # 3 = AND(a,b), 4 = NOT 3, 5 = NOT a, 6 = NOT b,
                  [(0, 3), (1, 3), (3, 4), (0, 5), (1, 6), (5, 7), (6, 7), (0, 8), (1, 8)], 3,   # 7 = OR(5,6), 8 = OR(a,b)
                  [[(3, False), (4, True), (7, True)], [(0, False), (5, True)], [(1, False), (6, True)]]),
    "xor_rebuilt": (["xmg", "xag"], [4, 3, 2, 3, 5, 2, 3],    # 3 = OR(a,b), 4 = AND(a,b), 5 = NOT 4, 6 = AND(3, 5);
                    [(0, 3), (1, 3), (0, 4), (1, 4), (4, 5), (3, 6), (5, 6), (0, 7), (1, 7), (7, 8), (0, 9), (2, 9)], 3,
                    [[(6, False), (7, False), (8, True)], [(4, False), (5, True)]]),   # 7 = XOR(a,b), 8 = NOT 7, 9 = AND(a,c)
    "majority": (["mig", "xmg"], [1, 3, 3, 3, 4, 4],          # 3 = MAJ(a,b,c) = OR(OR(AND ab, AND ac), AND bc) = 8
                 [(0, 3), (1, 3), (2, 3), (0, 4), (1, 4), (0, 5), (2, 5), (1, 6), (2, 6), (4, 7), (5, 7), (7, 8), (6, 8)], 3,
                 [[(3, False), (8, False)]]),
}
CONSTRUCTED_CASES = [(name, kind) for name, (kinds, *_) in CONSTRUCTED.items() for kind in kinds]


def oracle_classes(c, kind, **kw):
    return oracle_classes_of(c["x"][:, 1], c["edge_index"].T, kind, **kw)


@pytest.mark.parametrize("name,kind", CONSTRUCTED_CASES)
@pytest.mark.parametrize("exhaustive", [True, False])
def test_oracle_finds_constructed_equivalences(name, kind, exhaustive):
    _, codes, edges, n_pi, classes = CONSTRUCTED[name]
    c = circuit(codes, edges, n_pi)
    rep, comp = oracle_classes(c, kind, exhaustive=exhaustive, patterns=4096, seed=3)
    assert partition(rep, comp) == expected_partition(len(c["x"]), classes)


@pytest.mark.parametrize("kind,mix,exhaustive", [("aig", "aig", False), ("mig", "mig4", True), ("xmg", "xmg", False),
                                                 ("xag", "xag", True)])
def test_reference_words_give_the_oracle_counts(kind, mix, exhaustive):
    """The words of sim_classes_oracle are those oracle/logic_sim.simulate counts: same ones and pair distances."""
    import sim_classes_oracle as SO
    from deepgate import synth
    from oracle import logic_sim as OL
    c = synth.make_circuit(mix, 10 if exhaustive else 20, 300, seed=6, window=30)
    code, ei, pairs = c["x"][:, 1], c["edge_index"].T, c["tt_pair_index"].T
    kw = dict(patterns=64 * 7, seed=5, exhaustive=exhaustive)
    ones, diff, patterns = OL.simulate(code, ei, kind, pairs=pairs, **kw)
    net, p2 = SO._prepare(code, ei, kind, None, kw["patterns"], exhaustive)
    words = SO.pass_words(net, np.arange(patterns // 64), 5, exhaustive)
    assert p2 == patterns
    assert np.array_equal(OL.popcount(words), ones)
    assert np.array_equal(OL.popcount(words[pairs[0]] ^ words[pairs[1]]), diff)


def test_oracle_classes_do_not_depend_on_passes():
    from deepgate import synth
    c = synth.make_circuit("xmg", 20, 300, seed=5, window=30)
    one = oracle_classes(c, "xmg", patterns=64 * 13, seed=3)
    assert (np.bincount(one[0]) > 1).any()
    for step in (1, 3, 4):
        split = oracle_classes(c, "xmg", patterns=64 * 13, seed=3, words_per_pass=step)
        assert np.array_equal(one[0], split[0]) and np.array_equal(one[1], split[1])


def test_oracle_classes_keep_circuits_apart():
    """Two copies of one circuit in a batch: equal words, never one class."""
    _, codes, edges, n_pi, classes = CONSTRUCTED["de_morgan"]
    c = circuit(codes, edges, n_pi)
    n = len(c["x"])
    code = np.concatenate([c["x"][:, 1]] * 2)
    ei = np.concatenate([c["edge_index"], c["edge_index"] + n]).T
    rep, comp = oracle_classes_of(code, ei, "mig", batch=np.repeat([0, 1], n), exhaustive=True)
    shifted = [[(v + n, p) for v, p in cls] for cls in classes]
    assert partition(rep, comp) == expected_partition(2 * n, classes + shifted)


def test_class_pair_draw():
    from deepgate.simulate import _class_pairs_for, class_pair_count
    rep = np.array([0, 1, 0, 3, 1, 0, 6, 3, 0])              # classes {0, 2, 5, 8}, {1, 4}, {3, 7}: 6 + 1 + 1 pairs
    assert class_pair_count(rep) == 8
    every = _class_pairs_for(rep, 4, 100, seed=1)
    assert len(every) == 8 and len({tuple(p) for p in every}) == 8
    assert np.all(every[:, 0] < every[:, 1]) and np.all(rep[every[:, 0]] == rep[every[:, 1]])
    some = _class_pairs_for(rep, 4, 5, seed=1)
    assert len(some) == 5 and {tuple(p) for p in some} <= {tuple(p) for p in every}
    assert np.array_equal(some, _class_pairs_for(rep, 4, 5, seed=1))
    assert len(_class_pairs_for(np.arange(6), 0, 5, seed=1)) == 0
    big = np.zeros(3000, np.int64)                           # one class of 3000: 4 498 500 pairs
    draw = _class_pairs_for(big, 0, 1000, seed=2)
    assert len({tuple(p) for p in draw}) == 1000 and np.all(draw[:, 0] < draw[:, 1]) and draw.max() < 3000


def test_label_circuits_argument_errors_raise():
    import deepgate
    from deepgate import synth
    circuits = synth.make_circuits("mig", 2, 6, 30, cfg=72)
    for bad in (-1, 1.5, True):
        with pytest.raises(ValueError, match="class_pairs"):
            deepgate.label_circuits(circuits, "mig", "cpu", class_pairs=bad)
    with pytest.raises(ValueError, match="exceeds n_pairs"):
        deepgate.label_circuits(circuits, "mig", "cpu", n_pairs=8, class_pairs=9)
    G = deepgate.circuits_to_batch(circuits)
    with pytest.raises(RuntimeError, match="no CPU"):
        deepgate.equivalence_classes(G, "mig")
    with pytest.raises(ValueError, match="multiple of 64"):
        deepgate.equivalence_classes(G, "mig", patterns=100)
    with pytest.raises(ValueError, match="kind"):
        deepgate.equivalence_classes(G, "nand")


def test_cli_class_pairs_argument(tmp_path):
    from deepgate.simulate import main
    with pytest.raises(SystemExit):
        main(["--graphs", "g.npz", "--type", "mig", "--out", "d", "--class-pairs", "x"])
    with pytest.raises(SystemExit):
        main(["--graphs", "g.npz", "--type", "mig", "--out", "d", "--pairs", "8", "--class-pairs", "9"])
    with pytest.raises(FileNotFoundError):                   # parsed, then the missing input is opened
        main(["--graphs", str(tmp_path / "missing.npz"), "--type", "mig", "--out", str(tmp_path), "--class-pairs", "4"])


# ------------------------------------------------------------------ GPU
def gpu_classes(G, kind, **kw):
    import deepgate
    rep, comp, n_split = deepgate.equivalence_classes(G, kind, **kw)
    assert rep.device == G.edge_index.device and rep.dtype == torch.int64 and comp.dtype == torch.bool
    assert n_split == 0
    return rep.cpu().numpy(), comp.cpu().numpy()


def oracle_batch(G, kind, **kw):
    return oracle_classes_of(G.gate.reshape(-1).long().cpu().numpy(), G.edge_index.cpu().numpy(), kind,
                      batch=G.batch.cpu().numpy(), **kw)


def assert_same_classes(got, want):
    assert partition(*got) == partition(*want)
    assert (np.bincount(want[0]) > 1).any()                  # something to group


def constructed_for(kind):
    return [circuit(*CONSTRUCTED[name][1:4]) for name, k in CONSTRUCTED_CASES if k == kind]


MIXES = [("aig", "aig"), ("mig", "mig4"), ("xmg", "xmg"), ("xag", "xag")]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,mix", MIXES)
@pytest.mark.parametrize("depth", ["shallow", "deep"])
@pytest.mark.parametrize("exhaustive", [False, True])
def test_classes_match_oracle(kind, mix, depth, exhaustive):
    import deepgate
    from deepgate import synth
    if depth == "shallow":
        circuits = synth.make_circuits(mix, 6, (10, 16) if exhaustive else (16, 40), (100, 400), cfg=81, n_pairs=40)
    else:                                # window 3 over 3000 gates: > 1000 levels
        circuits = synth.make_circuits(mix, 2, 12, 3000, cfg=82, window=3, n_pairs=40)
    G = deepgate.circuits_to_batch(circuits + constructed_for(kind), "cuda")
    if depth == "deep":
        assert int(G.forward_level.max()) + 1 > 1000
    kw = dict(exhaustive=exhaustive, patterns=2048, seed=7)
    assert_same_classes(gpu_classes(G, kind, **kw), oracle_batch(G, kind, **kw))


@pytest.mark.gpu
@pytest.mark.parametrize("words,max_words", [(6, None), (13, None), (13, 4), (9, 8), (13, 12)])
def test_partial_slices_and_passes_match_oracle(words, max_words):
    """W not a multiple of the 4-word slice, and max_bytes small enough to force several passes."""
    import deepgate
    from deepgate import synth
    G = deepgate.circuits_to_batch(synth.make_circuits("xmg", 5, (16, 32), (200, 600), cfg=83, window=40, n_pairs=30), "cuda")
    n = G.x.size(0)
    kw = dict(patterns=64 * words, seed=123456789)
    got = gpu_classes(G, "xmg", max_bytes=2 ** 40 if max_words is None else 8 * n * max_words, **kw)
    assert_same_classes(got, oracle_batch(G, "xmg", **kw))


@pytest.mark.gpu
def test_cfg2_batch_matches_oracle():
    import deepgate
    from deepgate import synth
    G = deepgate.circuits_to_batch(synth.make_circuits("aig", 64, (16, 64), (500, 1500), cfg=2), "cuda")
    kw = dict(patterns=4096, seed=1)
    assert_same_classes(gpu_classes(G, "aig", **kw), oracle_batch(G, "aig", **kw))


@pytest.mark.gpu
def test_cfg5_100k_gate_mig_matches_oracle():
    import deepgate
    from deepgate import synth
    G = deepgate.circuits_to_batch(synth.make_circuits("mig", 1, 16, 100000, cfg=5, window=880), "cuda")
    kw = dict(patterns=4096, seed=2)
    assert_same_classes(gpu_classes(G, "mig", **kw), oracle_batch(G, "mig", **kw))


@pytest.mark.gpu
def test_circuit_classes_do_not_depend_on_the_batch():
    import deepgate
    from deepgate import synth
    circuits = synth.make_circuits("xag", 16, (16, 40), (100, 500), cfg=85, n_pairs=20)
    circuits[3] = circuits[9]                                # equal functions in two circuits of one batch
    alone = gpu_classes(deepgate.circuits_to_batch(circuits[9:10], "cuda"), "xag", patterns=1024, seed=4)
    batch = deepgate.circuits_to_batch(circuits, "cuda")
    rep, comp = gpu_classes(batch, "xag", patterns=1024, seed=4)
    ptr = batch.ptr.cpu().numpy()
    for i in (3, 9):
        lo, hi = int(ptr[i]), int(ptr[i + 1])
        assert partition(rep[lo:hi] - lo, comp[lo:hi]) == partition(*alone)
    circuit_of = batch.batch.cpu().numpy()
    assert np.array_equal(circuit_of[rep], circuit_of)       # no class spans two circuits


@pytest.mark.gpu
@pytest.mark.parametrize("passes", [1, 2])
def test_verification_splits_exactly_the_wrong_members(passes):
    """Feeds mgv_sim_classes_verify_pass a class assignment with known wrong members (bad input to a checked entry
    point) and checks that mgv_sim_classes_split makes exactly those singletons."""
    import deepgate
    from deepgate import _native as nat, synth
    from deepgate.simulate import _Sim, _circuit_ids
    circuits = synth.make_circuits("xmg", 4, (10, 16), (100, 300), cfg=87)
    G = deepgate.circuits_to_batch(circuits, "cuda")
    rep, comp, n_split = deepgate.equivalence_classes(G, "xmg", patterns=1024, seed=6)
    assert n_split == 0
    r, c = rep.cpu().numpy(), comp.cpu().numpy().astype(np.uint8)
    ptr = G.ptr.cpu().numpy()
    n = len(r)
    wrong = {}
    members = [v for v in range(int(ptr[0]), int(ptr[1])) if r[v] != v]
    v = members[0]
    wrong[v] = (r[v], 1 - c[v])                              # a true member with the wrong polarity
    v = members[1]
    wrong[v] = (next(u for u in range(int(ptr[2]), int(ptr[3])) if r[u] == u), c[v])     # a representative in another circuit
    v = members[2]
    wrong[v] = (n + 5, c[v])                                 # representative outside [0, N)
    singles = [u for u in range(int(ptr[1]), int(ptr[2])) if r[u] == u and np.sum(r == u) == 1]
    wrong[singles[-1]] = (singles[0], 0)                      # a different function of the same circuit
    wrong[singles[-2]] = (singles[-2], 1)                     # a representative marked complemented
    assert len(wrong) == 5
    bad_rep, bad_comp = r.copy(), c.copy()
    for v, (rr, cc) in wrong.items():
        bad_rep[v], bad_comp[v] = rr, cc
    dev = G.edge_index.device
    rep_t = torch.from_numpy(bad_rep).to(dev)
    comp_t = torch.from_numpy(bad_comp).to(dev)
    bad = torch.zeros(n, dtype=torch.uint8, device=dev)
    circuit = _circuit_ids(G, n, dev).to(torch.int32).contiguous()
    lib = nat.lib()
    st = nat.stream_of(dev)
    s = _Sim(G, "xmg", 1024, 6, False, 8 * n * (16 if passes == 1 else 8))
    W = s.words_per_pass()
    sim = nat.workspace(lib.mgv_logic_sim_bytes(n, W), dev)
    ones = torch.zeros(n, dtype=torch.int64, device=dev)
    count = 0
    for _, w in s.passes(lib, st, W, sim, ones, None, 0, None):
        nat.check(lib.mgv_sim_classes_verify_pass(nat.ptr(sim), n, w, nat.ptr(circuit), nat.ptr(rep_t), nat.ptr(comp_t),
                                                  nat.ptr(bad), st), "mgv_sim_classes_verify_pass")
        count += 1
    assert count == passes
    ws = nat.workspace(8, dev)
    n_split = ctypes.c_int64(-1)
    nat.check(lib.mgv_sim_classes_split(n, nat.ptr(rep_t), nat.ptr(comp_t), nat.ptr(bad), nat.ptr(ws), ws.numel(),
                                        ctypes.byref(n_split), st), "mgv_sim_classes_split")
    assert n_split.value == len(wrong)
    assert set(np.flatnonzero(bad.cpu().numpy()).tolist()) == set(wrong)
    want_rep, want_comp = bad_rep.copy(), bad_comp.copy()
    for v in wrong:
        want_rep[v], want_comp[v] = v, 0
    assert np.array_equal(rep_t.cpu().numpy(), want_rep) and np.array_equal(comp_t.cpu().numpy(), want_comp)
    with pytest.raises(RuntimeError, match="NULL bad"):
        nat.check(lib.mgv_sim_classes_verify_pass(nat.ptr(sim), n, W, nat.ptr(circuit), nat.ptr(rep_t), nat.ptr(comp_t),
                                                  None, st), "mgv_sim_classes_verify_pass")


@pytest.mark.gpu
def test_label_circuits_with_class_pairs_end_to_end(tmp_path):
    import types
    import deepgate
    from deepgate import synth
    from deepgate.simulate import class_pair_count
    circuits = synth.make_circuits("mig4", 24, (8, 16), (40, 120), cfg=86, window=16)
    for c in circuits:
        c.pop("tt_pair_index")
    kw = dict(batch_size=10, n_pairs=16, patterns=2048, seed=5)
    labelled = deepgate.label_circuits(circuits, "mig", "cuda:0", class_pairs=6, **kw)
    again = deepgate.label_circuits(circuits, "mig", "cuda:0", class_pairs=6, **kw)
    drawn = 0
    for i, (c, d) in enumerate(zip(labelled, again)):
        assert np.array_equal(c["tt_pair_index"], d["tt_pair_index"]) and np.array_equal(c["tt_sim"], d["tt_sim"])
        assert np.array_equal(c["prob"], d["prob"])
        rep, comp, n_split = deepgate.equivalence_classes(deepgate.circuits_to_batch([c], "cuda"), "mig", patterns=2048, seed=5)
        rep, comp = rep.cpu().numpy(), comp.cpu().numpy()
        k = min(6, class_pair_count(rep))
        tpi, tt = c["tt_pair_index"], c["tt_sim"]
        assert len(tpi) == 16 and np.all(tpi[:, 0] != tpi[:, 1])
        a, b = tpi[:k, 0], tpi[:k, 1]
        assert np.all(rep[a] == rep[b])                       # the class pairs come first ...
        assert np.array_equal(tt[:k], (comp[a] != comp[b]).astype(np.float32))   # ... labelled exactly 0 or 1
        assert len({tuple(p) for p in tpi[:k]}) == k
        drawn += k
    assert drawn > 24
    plain = deepgate.label_circuits(circuits, "mig", "cuda:0", **kw)
    zero = deepgate.label_circuits(circuits, "mig", "cuda:0", class_pairs=0, **kw)
    for p, z in zip(plain, zero):
        assert set(p) == set(z) and all(np.array_equal(p[key], z[key]) for key in p)
    root = str(tmp_path / "ds")
    os.makedirs(root)
    gp, lp = deepgate.write_npz(labelled, os.path.join(root, "graphs.npz"), os.path.join(root, "labels.npz"), "mig")
    torch.manual_seed(0)
    train, val = deepgate.NpzParser(root, gp, lp, "mig").get_dataset()
    enc = deepgate.digae_layer.DirectMultiGCNEncoder(dim_hidden=64, dim_feature=6, s_rounds=1, t_rounds=1)
    model = deepgate.dg_ae_model_mig.Model(struct_encoder=enc, dim_hidden=64)
    args = types.SimpleNamespace(model="DG_AE", type="mig")
    trainer = deepgate.Trainer(args, model, training_id="simcls", save_dir=str(tmp_path / "exp"), device="cuda:0",
                               batch_size=4, distributed=False, rc_prob_func_weight=[1.0, 4.0, 4.0])
    trainer.train(1, train, val)
    log = open(trainer.log_path).read()
    assert "train|" in log and "nan" not in log.lower()
