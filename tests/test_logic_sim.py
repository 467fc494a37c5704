"""Circuit labelling by logic simulation (deepgate.simulate, csrc/logic_sim.cu) against the numpy simulator
oracle/logic_sim.py.  CPU: closed forms of the oracle, pass splitting, the npz writer through NpzParser, argument errors.
GPU: counts bit-equal to the oracle over gate mixes, modes, depths, pass splits, schedules and batch placement; input
validation; labels -> npz -> NpzParser -> one training epoch."""
import os

import numpy as np
import pytest
import torch

from oracle import logic_sim as OL


def circuit(codes, edges, n_pi):
    """A hand-built circuit dict: ``n_pi`` INPUTs, then gates with ``codes``; ``edges`` (src, dst) pairs."""
    code = np.array([0] * n_pi + list(codes), dtype=np.int64)
    x = np.stack([np.arange(code.size), code], axis=1)
    ei = np.array(edges, dtype=np.int64).reshape(-1, 2)
    return {"x": x, "edge_index": ei, "prob": np.zeros(code.size, np.float32),
            "tt_pair_index": np.zeros((0, 2), np.int64), "tt_sim": np.zeros(0, np.float32)}


def oracle_of(c, kind, pairs=None, **kw):
    return OL.simulate(c["x"][:, 1], c["edge_index"].T, kind, pairs=None if pairs is None else np.asarray(pairs).T, **kw)


# (kind, gate codes after the inputs, edges, inputs, pairs, expected prob of the last node, expected distances)
CLOSED_FORMS = [
    ("aig", [1], [(0, 2), (1, 2)], 2, [(0, 0), (0, 1)], 0.25, [0.0, 0.5]),           # AND2
    ("aig", [1, 2], [(0, 2), (1, 2), (2, 3)], 2, [(2, 3)], 0.75, [1.0]),              # NOT(AND2); x vs NOT x
    ("mig", [3], [(0, 2), (1, 2)], 2, [(0, 1)], 0.25, [0.5]),                          # AND2
    ("mig", [4], [(0, 2), (1, 2)], 2, [(2, 2)], 0.75, [0.0]),                          # OR2
    ("xag", [5], [(0, 2), (1, 2)], 2, [(0, 1)], 0.5, [0.5]),                           # XOR2
    ("mig", [1], [(0, 3), (1, 3), (2, 3)], 3, [(1, 2)], 0.5, [0.5]),                   # MAJ3
    ("xmg", [3, 2], [(0, 2), (1, 2), (2, 3)], 2, [(2, 3)], 0.75, [1.0]),               # NOT(AND2)
]


@pytest.mark.parametrize("case", range(len(CLOSED_FORMS)))
def test_oracle_closed_forms_exhaustive(case):
    kind, codes, edges, n_pi, pairs, p_last, dist = CLOSED_FORMS[case]
    c = circuit(codes, edges, n_pi)
    ones, diff, patterns = oracle_of(c, kind, pairs, exhaustive=True)
    assert patterns == 64
    assert ones[-1] / patterns == p_last
    assert np.all(ones[:n_pi] * 2 == patterns)                                   # every INPUT is 1 half the time
    assert list(diff / patterns) == dist


def test_oracle_exhaustive_covers_every_assignment():
    """8 inputs: 256 patterns, AND of all 8 is 1 exactly once."""
    c = circuit([3], [(i, 8) for i in range(8)], 8)
    ones, _, patterns = oracle_of(c, "mig", exhaustive=True)
    assert patterns == 256 and ones[-1] == 1


@pytest.mark.parametrize("exhaustive", [False, True])
def test_oracle_counts_do_not_depend_on_passes(exhaustive):
    from deepgate import synth
    c = synth.make_circuit("xmg", 9 if exhaustive else 20, 300, seed=5, window=30)
    pairs = c["tt_pair_index"]
    kw = dict(exhaustive=exhaustive, patterns=64 * 13, seed=3)
    one = oracle_of(c, "xmg", pairs, **kw)
    for step in (1, 3, 4):
        split = oracle_of(c, "xmg", pairs, words_per_pass=step, **kw)
        assert np.array_equal(one[0], split[0]) and np.array_equal(one[1], split[1])


def test_oracle_random_inputs_are_the_stated_hash():
    w = OL.input_words([0, 5], [0, 7], seed=11, exhaustive=False)
    mix = lambda z: OL.mix(np.array([z], np.uint64))[0]
    assert w[1, 1] == mix(mix(np.uint64(11)) ^ np.uint64((5 << 40) | 7))
    e = OL.input_words([0, 1, 6], [0, 1], seed=0, exhaustive=True)
    assert e[0, 0] == np.uint64(0xAAAAAAAAAAAAAAAA) and e[1, 1] == np.uint64(0xCCCCCCCCCCCCCCCC)
    assert e[2, 0] == 0 and e[2, 1] == np.uint64(0xFFFFFFFFFFFFFFFF)


@pytest.mark.parametrize("kind,mix", [("aig", "aig"), ("xmg", "xmg")])
def test_write_npz_round_trips_through_npz_parser(tmp_path, kind, mix):
    import deepgate
    from deepgate import synth
    circuits = synth.make_circuits(mix, 6, 6, 40, cfg=71, window=12, n_pairs=8)
    for i, c in enumerate(circuits):                    # labels as label_circuits returns them (float32 prob / distance)
        c["prob"] = np.random.default_rng(i).random(len(c["x"])).astype(np.float32)
        c["tt_sim"] = np.random.default_rng(100 + i).random(8).astype(np.float32)
    root = str(tmp_path / "ds")
    os.makedirs(root)
    gp, lp = deepgate.write_npz(circuits, os.path.join(root, "graphs.npz"),
                                None if kind == "aig" else os.path.join(root, "labels.npz"), kind)
    parser = deepgate.NpzParser(root, gp, lp, kind, random_shuffle=False, trainval_split=1.0)
    graphs = parser.train_dataset.graphs
    assert len(graphs) == len(circuits)
    for c, g in zip(circuits, graphs):
        assert torch.equal(g.prob.reshape(-1), torch.from_numpy(c["prob"]))
        assert torch.equal(g.tt_pair_index, torch.from_numpy(c["tt_pair_index"].T.copy()))
        assert torch.equal(g.tt_sim, torch.from_numpy(c["tt_sim"]))
        assert torch.equal(g.edge_index, torch.from_numpy(c["edge_index"].T.copy()))
        assert torch.equal(g.gate.reshape(-1).long(), torch.from_numpy(c["x"][:, 1]))


def test_argument_errors_raise():
    import deepgate
    from deepgate import synth
    G = deepgate.circuits_to_batch(synth.make_circuits("mig", 2, 6, 30, cfg=72))
    with pytest.raises(RuntimeError, match="no CPU"):
        deepgate.simulate(G, "mig")
    with pytest.raises(ValueError, match="multiple of 64"):
        deepgate.simulate(G, "mig", patterns=100)
    with pytest.raises(ValueError, match="kind"):
        deepgate.simulate(G, "nand")
    big = deepgate.circuits_to_batch(synth.make_circuits("mig", 1, 25, 30, cfg=73))
    with pytest.raises(ValueError, match="25 inputs"):
        deepgate.simulate(big, "mig", exhaustive=True)


def test_cli_arguments():
    from deepgate.simulate import main
    with pytest.raises(SystemExit):
        main(["--graphs", "g.npz", "--type", "nand", "--out", "d"])


# ------------------------------------------------------------------ GPU
def gpu_counts(G, kind, **kw):
    from deepgate.simulate import simulate_counts
    ones, diff, patterns = simulate_counts(G, kind, **kw)
    return ones.cpu().numpy(), diff.cpu().numpy(), patterns


def oracle_batch(G, kind, **kw):
    return OL.simulate(G.gate.reshape(-1).long().cpu().numpy(), G.edge_index.cpu().numpy(), kind,
                       batch=G.batch.cpu().numpy(), pairs=G.tt_pair_index.cpu().numpy(), **kw)


def assert_same(got, want):
    assert got[2] == want[2]
    assert np.array_equal(got[0], want[0]), int(np.flatnonzero(got[0] != want[0])[0])
    assert np.array_equal(got[1], want[1])


MIXES = [("aig", "aig"), ("mig", "mig4"), ("xmg", "xmg"), ("xag", "xag")]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,mix", MIXES)
@pytest.mark.parametrize("depth", ["shallow", "deep"])
@pytest.mark.parametrize("exhaustive", [False, True])
def test_counts_match_oracle(kind, mix, depth, exhaustive):
    import deepgate
    from deepgate import synth
    if depth == "shallow":
        circuits = synth.make_circuits(mix, 6, (10, 16) if exhaustive else (16, 40), (100, 400), cfg=81, n_pairs=40)
    else:                                # window 3 over 3000 gates: > 1000 levels
        circuits = synth.make_circuits(mix, 2, 12, 3000, cfg=82, window=3, n_pairs=40)
    G = deepgate.circuits_to_batch(circuits, "cuda")
    if depth == "deep":
        assert int(G.forward_level.max()) + 1 > 1000
    kw = dict(exhaustive=exhaustive, patterns=2048, seed=7)
    assert_same(gpu_counts(G, kind, **kw), oracle_batch(G, kind, **kw))


@pytest.mark.gpu
@pytest.mark.parametrize("words,max_words", [(6, None), (13, None), (13, 4), (9, 8)])
def test_partial_slices_and_passes_match_oracle(words, max_words):
    """W not a multiple of the 4-word slice, and max_bytes small enough to force several passes."""
    import deepgate
    from deepgate import synth
    G = deepgate.circuits_to_batch(synth.make_circuits("xmg", 5, (16, 32), (200, 600), cfg=83, window=40, n_pairs=30), "cuda")
    n = G.x.size(0)
    kw = dict(patterns=64 * words, seed=123456789)
    got = gpu_counts(G, "xmg", max_bytes=2 ** 40 if max_words is None else 8 * n * max_words, **kw)
    assert_same(got, oracle_batch(G, "xmg", **kw))


@pytest.mark.gpu
def test_cfg2_batch_matches_oracle():
    import deepgate
    from deepgate import synth
    G = deepgate.circuits_to_batch(synth.make_circuits("aig", 64, (16, 64), (500, 1500), cfg=2), "cuda")
    kw = dict(patterns=4096, seed=1)
    assert_same(gpu_counts(G, "aig", **kw), oracle_batch(G, "aig", **kw))


@pytest.mark.gpu
def test_cfg5_100k_gate_mig_matches_oracle():
    import deepgate
    from deepgate import synth
    G = deepgate.circuits_to_batch(synth.make_circuits("mig", 1, 16, 100000, cfg=5, window=880), "cuda")
    assert int(G.forward_level.max()) + 1 >= 600
    kw = dict(patterns=4096, seed=2)
    assert_same(gpu_counts(G, "mig", **kw), oracle_batch(G, "mig", **kw))


@pytest.mark.gpu
def test_two_stream_host_schedule_equals_device_schedule(monkeypatch):
    import deepgate
    from deepgate import synth
    circuits = synth.make_circuits("mig4", 7, (16, 40), (300, 900), cfg=84, n_pairs=50)
    G = deepgate.circuits_to_batch(circuits, "cuda")
    assert G.sweep_streams == 2 and G.sched_order.is_cuda
    host = gpu_counts(G, "mig", patterns=1024, seed=9)
    assert deepgate.schedule.schedule_for_batch(G).streams == 2            # the batch's own cached schedule was used
    monkeypatch.setenv("MGV_DEVICE_SCHEDULE", "1")
    D = deepgate.circuits_to_batch(circuits, "cuda")
    dev = gpu_counts(D, "mig", patterns=1024, seed=9)
    assert_same(host, dev)


@pytest.mark.gpu
def test_circuit_labels_do_not_depend_on_the_batch():
    import deepgate
    from deepgate import synth
    circuits = synth.make_circuits("xag", 16, (16, 40), (100, 500), cfg=85, n_pairs=20)
    alone = deepgate.simulate(deepgate.circuits_to_batch(circuits[9:10], "cuda"), "xag", patterns=1024, seed=4)
    batch = deepgate.circuits_to_batch(circuits, "cuda")
    together = deepgate.simulate(batch, "xag", patterns=1024, seed=4)
    lo, hi = int(batch.ptr[9]), int(batch.ptr[10])
    assert torch.equal(together[0][lo:hi], alone[0])
    assert torch.equal(together[1][9 * 20:10 * 20], alone[1])


BAD = [  # (kind, codes, edges, n_pi, pairs, message)
    ("mig", [1], [(0, 2), (1, 2)], 2, [], "node 2 .*MAJ needs fan-in 3"),
    ("mig", [2], [(0, 2), (1, 2)], 2, [], "node 2 .*NOT needs fan-in 1"),
    ("xag", [3, 5], [(0, 2), (1, 2), (2, 3)], 2, [], "node 3 .*AND / OR / XOR need fan-in >= 2"),
    ("mig", [4, 3], [(0, 2), (0, 3), (1, 3)], 2, [], "node 2 .*fan-in 1.*AND / OR / XOR"),
    ("aig", [1, 3], [(0, 2), (1, 2), (0, 3), (1, 3)], 2, [], "node 3 .*code 3.*not defined"),
    ("mig", [3, 3], [(0, 2), (1, 2)], 2, [], "node 3 .*fan-in 0"),
    ("mig", [3, 0], [(0, 2), (1, 2), (2, 3)], 2, [], "node 3 .*INPUT with predecessors"),
    ("mig", [3], [(0, 2), (1, 2)], 2, [(0, 3)], "pair 0 .*outside"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", range(len(BAD)))
def test_validation_names_the_node(case):
    import deepgate
    kind, codes, edges, n_pi, pairs, msg = BAD[case]
    c = circuit(codes, edges, n_pi)
    G = deepgate.circuits_to_batch([c], "cuda")
    if pairs:
        G.tt_pair_index = torch.tensor(pairs, device="cuda").T.contiguous()
    with pytest.raises(RuntimeError, match=msg):
        deepgate.simulate(G, kind)


@pytest.mark.gpu
def test_label_write_parse_train_end_to_end(tmp_path):
    import types
    import deepgate
    from deepgate import synth
    circuits = synth.make_circuits("mig4", 24, (8, 16), (40, 120), cfg=86, window=16)
    for c in circuits:
        c.pop("tt_pair_index")
    labelled = deepgate.label_circuits(circuits, "mig", "cuda:0", batch_size=10, n_pairs=16, patterns=2048, seed=5)
    assert all(len(c["tt_pair_index"]) == 16 and np.all(c["tt_pair_index"][:, 0] != c["tt_pair_index"][:, 1]) for c in labelled)
    G = deepgate.circuits_to_batch(labelled[:1], "cuda")
    want = oracle_batch(G, "mig", patterns=2048, seed=5)
    assert np.array_equal(labelled[0]["prob"], (want[0] / 2048).astype(np.float32))
    assert np.array_equal(labelled[0]["tt_sim"], (want[1] / 2048).astype(np.float32))
    root = str(tmp_path / "ds")
    os.makedirs(root)
    gp, lp = deepgate.write_npz(labelled, os.path.join(root, "graphs.npz"), os.path.join(root, "labels.npz"), "mig")
    torch.manual_seed(0)
    train, val = deepgate.NpzParser(root, gp, lp, "mig").get_dataset()
    enc = deepgate.digae_layer.DirectMultiGCNEncoder(dim_hidden=64, dim_feature=6, s_rounds=1, t_rounds=1)
    model = deepgate.dg_ae_model_mig.Model(struct_encoder=enc, dim_hidden=64)
    args = types.SimpleNamespace(model="DG_AE", type="mig")
    trainer = deepgate.Trainer(args, model, training_id="sim", save_dir=str(tmp_path / "exp"), device="cuda:0",
                               batch_size=4, distributed=False, rc_prob_func_weight=[1.0, 4.0, 4.0])
    status = trainer.train_step(next(iter(deepgate.DataLoader(train, batch_size=4))).to("cuda:0"))
    assert all(torch.isfinite(status[k]).all() for k in ("recon_loss", "prob_loss", "func_loss"))
    trainer.train(1, train, val)
    log = open(trainer.log_path).read()
    assert "train|" in log and "nan" not in log.lower()
