"""AIG -> MIG / XMG / XAG mapping (deepgate/mapping.py, csrc/map_cuts.cu).
CPU: the match tables exhaustively; the reference mapping (tests/map_oracle.py + mapping.emit) keeps every node's and
every output's function, node order, NOT sharing and edge order; adders give the full-adder gates; input errors.
GPU: the per-node arrays are bit-equal to the reference; mapped copies simulate equal to their origins at scale; a
circuit maps the same alone and in a batch; ``--aiger --type xmg --map`` goes through NpzParser and one training epoch."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import map_oracle as MO
import test_aiger as TA
from deepgate import mapping as MP
from deepgate import synth
from deepgate.aiger import read_aiger
from deepgate.simulate import CODE_TABLES

KINDS = ("mig", "xmg", "xag")
CODES = CODE_TABLES["xmg"]
# outputs 8 = AND(a, AND(NOT a, b)) = 0, 15 = (a AND b) OR (a AND NOT b) = a, 16 = AND(15, b): an AND over an alias
FOLDS = "aag 9 2 0 3 6\n2\n4\n8\n15\n16\n6 3 4\n8 2 6\n10 2 4\n12 2 5\n14 11 13\n16 15 4\n"
TEXTS = dict(TA.FIXTURES, folds=FOLDS, adder4=TA.adder(4), mult3=TA.multiplier(3), mult4=TA.multiplier(4))


def circuit(tmp_path, name, text):
    return read_aiger(TA.write(tmp_path, name + ".aag", text), "aig")


def gate_arity_counts(m):
    """{(code name, fan-in): count} of the gates of a mapped dict."""
    code = m["x"][:, 1]
    deg = np.bincount(m["edge_index"][:, 1], minlength=len(code))
    out = {}
    for c, d in zip(code.tolist(), deg.tolist()):
        if CODES[c] not in ("INPUT", "NOT"):
            out[(CODES[c], d)] = out.get((CODES[c], d), 0) + 1
    return out


def assert_well_formed(c, m, kind):
    """Node order, NOT sharing, inputs in place, (dst, src) edge order, gate codes and fan-ins of the library."""
    code, ei, origin = m["x"][:, 1], m["edge_index"], m["origin"]
    assert np.array_equal(m["x"][:, 0], np.arange(len(code)))
    assert np.array_equal(ei, ei[np.lexsort((ei[:, 0], ei[:, 1]))]) and np.all(ei[:, 0] < ei[:, 1])
    inputs = np.flatnonzero(c["x"][:, 1] == 0)
    k = inputs.size
    assert np.array_equal(code[:k], np.zeros(k)) and np.array_equal(origin[:k], 2 * inputs) and (code[k:] != 0).all()
    deg = np.bincount(ei[:, 1], minlength=len(code))
    allowed = {"AND": {2}, "OR": {2}, "XOR": {2, 3}, "MAJ": {3}, "NOT": {1}}
    lib = set(MP.LIBRARY[kind])
    allowed_names = {MP._CODE_NAME[g] for g in lib} | {"NOT"}
    for v in range(k, len(code)):
        name = CODES[code[v]]
        assert name in allowed_names and deg[v] in allowed[name], (v, name, deg[v])
        if name == "XOR":
            assert ("XOR%d" % deg[v]) in lib
    nots = np.flatnonzero(code == 2)
    src = np.zeros(len(code), np.int64)
    src[ei[:, 1]] = ei[:, 0]
    assert np.unique(src[nots]).size == nots.size                        # one NOT per node
    assert np.all(origin[nots] == origin[src[nots]] ^ 1)
    in_nots = nots[src[nots] < k]
    assert np.array_equal(in_nots, k + np.arange(in_nots.size)) and np.all(np.diff(src[in_nots]) > 0)
    rest = np.arange(k + in_nots.size, len(code))
    gates = rest[code[rest] != 2]
    assert np.all(np.diff(origin[gates] >> 1) > 0)                       # by the id of the AND they replace
    assert np.all(src[rest[code[rest] == 2]] == rest[code[rest] == 2] - 1)   # a gate's NOT directly follows it


def assert_equivalent(c, m, kind, text=None):
    """Every mapped node equals its origin literal on every input assignment; every output equals the file's."""
    orig = TA.node_words(c, "aig")
    words = TA.node_words(m, kind)
    o = m["origin"]
    assert np.array_equal(words, orig[o >> 1] ^ (o & 1)[:, None].astype(bool))
    if text is not None:
        value, _ = TA.evaluate(text)
        I, L, O, B, C, inputs, latches, outputs, ands, _ = TA.parse_aag(text)
        outs = outputs[:O] + [l[1] for l in latches] + outputs[O:]
        assert len(m["outputs"]) == len(outs)
        for lit, got in zip(outs, m["outputs"]):
            assert np.array_equal(TA.literal_bits(m, words, int(got), need_not_node=True), value(lit)), lit


# ------------------------------------------------------------------ CPU
@pytest.mark.parametrize("kind", KINDS)
def test_match_table_reproduces_every_table(kind):
    table = MP.MATCH[kind]
    sizes = {}
    for tt in range(256):
        if table[tt] < 0:
            continue
        gate, mask, out = MP.decode_match(int(table[tt]))
        assert gate in MP.LIBRARY[kind]
        assert MP._gate_table(gate, mask, out) == tt
        cls = {"AND2": "ANDOR", "OR2": "ANDOR"}.get(gate, gate)
        sizes[cls] = sizes.get(cls, 0) + 1
    want = {"mig": {"ANDOR": 8, "MAJ3": 8}, "xag": {"ANDOR": 8, "XOR2": 2},
            "xmg": {"ANDOR": 8, "XOR2": 2, "MAJ3": 8, "XOR3": 2}}[kind]
    assert sizes == want
    or_gate = ("AND2", 3, 1) if kind == "xag" else ("OR2", 0, 0)          # a OR b
    assert MP.decode_match(int(table[0xEE])) == or_gate


@pytest.mark.parametrize("kind", KINDS)
def test_reference_mapping_keeps_every_function(tmp_path, kind):
    for name, text in sorted(TEXTS.items()):
        c = circuit(tmp_path, name, text)
        m = MO.map_circuit(c, kind)
        assert_well_formed(c, m, kind)
        assert_equivalent(c, m, kind, text)
        assert sum(gate_arity_counts(m).values()) <= int((c["x"][:, 1] == 1).sum()), name


def test_constants_and_aliases_fold(tmp_path):
    c = circuit(tmp_path, "folds", FOLDS)
    assert int((c["x"][:, 1] == 1).sum()) == 6                # read_aiger folds none of them
    for kind in KINDS:
        m = MO.map_circuit(c, kind)
        # output 8 is constant 0, output 15 is input a; 16 = AND(a, b) stays, one AND2
        assert m["outputs"].tolist()[:2] == [-2, 0]
        assert gate_arity_counts(m) == {("AND", 2): 1}


@pytest.mark.parametrize("kind", KINDS)
def test_synthetic_aigs_with_double_negation(kind):
    for c in synth.make_circuits("aig", 12, (6, 12), (30, 300), cfg=91, window=8):
        m = MO.map_circuit(c, kind)
        assert_well_formed(c, m, kind)
        assert_equivalent(c, m, kind)
        assert len(m["outputs"]) == len(MP._roots(c))
    nn = [c for c in synth.make_circuits("aig", 12, (6, 12), (30, 300), cfg=91, window=8)
          if ((c["x"][c["edge_index"][:, 0], 1] == 2) & (c["x"][c["edge_index"][:, 1], 1] == 2)).any()]
    assert nn                                                  # the set does contain NOT-of-NOT chains


@pytest.mark.parametrize("n", range(2, 9))
def test_adders_map_to_full_adder_gates(tmp_path, n):
    c = circuit(tmp_path, "adder%d" % n, TA.adder(n))
    assert gate_arity_counts(MO.map_circuit(c, "xmg")) == {("XOR", 3): n - 1, ("MAJ", 3): n - 1, ("XOR", 2): 1,
                                                            ("AND", 2): 1}
    assert gate_arity_counts(MO.map_circuit(c, "mig")).get(("MAJ", 3)) == n - 1
    assert gate_arity_counts(MO.map_circuit(c, "xag")).get(("XOR", 2)) == 2 * n - 1


@pytest.mark.parametrize("n", range(2, 9))
def test_multipliers_use_no_more_gates_than_ands(tmp_path, n):
    c = circuit(tmp_path, "mult%d" % n, TA.multiplier(n))
    for kind in KINDS:
        assert sum(gate_arity_counts(MO.map_circuit(c, kind)).values()) <= int((c["x"][:, 1] == 1).sum())


def _aig(x_codes, edges, name="bad"):
    return {"x": np.stack([np.arange(len(x_codes)), x_codes], axis=1), "edge_index": np.array(edges, np.int64).reshape(-1, 2),
            "name": name}


@pytest.mark.parametrize("case,msg", [
    (_aig([0, 0, 3], [[0, 2], [1, 2]]), "bad: node 2 has gate code 3"),
    (_aig([0, 0, 1], [[0, 2]]), "bad: node 2 \\(AND\\) has fan-in 1, needs 2"),
    (_aig([0, 0, 0, 1], [[0, 3], [1, 3], [2, 3]]), "bad: node 3 \\(AND\\) has fan-in 3, needs 2"),
    (_aig([0, 0, 2], [[0, 2], [1, 2]]), "bad: node 2 \\(NOT\\) has fan-in 2, needs 1"),
    (_aig([0, 0, 1], [[0, 1], [0, 2], [1, 2]]), "bad: node 1 \\(INPUT\\) has fan-in 1, needs 0"),
    (_aig([0, 1, 0], [[0, 1], [2, 1]]), "bad: edge 1 \\(2 -> 1\\)"),
    (_aig([0, 0, 1], [[0, 2], [2, 2]]), "bad: edge 1 \\(2 -> 2\\)"),
])
def test_input_errors_name_circuit_and_place(case, msg):
    good = _aig([0, 0, 1], [[0, 2], [1, 2]], "good")
    with pytest.raises(ValueError, match="^" + msg):
        MP.map_circuits([good, case], "xmg", "cuda:0")


def test_kind_and_device_errors():
    good = _aig([0, 0, 1], [[0, 2], [1, 2]], "good")
    for kind in ("aig", "nand"):
        with pytest.raises(ValueError, match="kind"):
            MP.map_circuits([good], kind, "cuda:0")
    with pytest.raises(ValueError, match="CUDA"):
        MP.map_circuits([good], "xmg", "cpu")


def test_cli_map_arguments():
    from deepgate.simulate import main
    with pytest.raises(SystemExit):
        main(["--graphs", "g.npz", "--type", "xmg", "--map", "--out", "d"])
    with pytest.raises(SystemExit):
        main(["--aiger", "a.aag", "--type", "aig", "--map", "--out", "d"])


# ------------------------------------------------------------------ GPU
def _cases(tmp_path):
    out = [circuit(tmp_path, name, text) for name, text in sorted(TEXTS.items())]
    for n in range(2, 9):
        out += [circuit(tmp_path, "adder%d" % n, TA.adder(n)), circuit(tmp_path, "mult%d" % n, TA.multiplier(n))]
    out += synth.make_circuits("aig", 160, (8, 64), (50, 2000), cfg=92)
    out += synth.make_circuits("aig", 96, (8, 32), (200, 2000), cfg=93, window=6)        # deep
    out += synth.make_circuits("aig", 64, (3, 8), (20, 300), cfg=94, window=3)           # narrow: many folds
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_node_arrays_equal_reference(tmp_path, kind):
    circuits = _cases(tmp_path)
    n_alias = 0
    for i0 in range(0, len(circuits), 64):
        chunk = circuits[i0:i0 + 64]
        for j, (c, got) in enumerate(zip(chunk, MP._node_arrays(chunk, kind, "cuda:0"))):
            want = MO.node_arrays(c, kind)
            for key in ("required", "best", "match", "flow", "alias"):
                assert np.array_equal(got[key], want[key]), (i0 + j, key)
            n_alias += int((want["alias"] != MP.NO_ALIAS).sum())
    assert n_alias > 0


def _as_kind(c, kind):
    """An AIG dict in the codes of ``kind`` (AND 1 -> 3), so it can share a batch with its mapped copy."""
    x = np.array(c["x"], copy=True)
    x[:, 1] = np.array([0, CODES.index("AND"), CODES.index("NOT")])[x[:, 1]]
    return {"x": x, "edge_index": c["edge_index"]}


def _check_pairs(circuits, kind):
    import deepgate
    mapped = MP.map_circuits(circuits, kind, "cuda:0")
    both = [_as_kind(c, kind) for c in circuits] + [{"x": m["x"], "edge_index": m["edge_index"]} for m in mapped]
    sizes = [len(c["x"]) for c in both]
    start = np.concatenate([[0], np.cumsum(sizes)])
    pairs, flip, orig_out, const_out = [], [], [], []
    for i, (c, m) in enumerate(zip(circuits, mapped)):
        a, b = start[i], start[len(circuits) + i]
        o = m["origin"]
        pairs.append(np.stack([a + (o >> 1), b + np.arange(len(o))], axis=1))
        flip.append(o & 1)
        roots = np.asarray(c["outputs"]) if "outputs" in c else 2 * MP._roots(c)
        keep = (roots >= 0) & (m["outputs"] >= 0)
        pairs.append(np.stack([a + (roots[keep] >> 1), b + (m["outputs"][keep] >> 1)], axis=1))
        flip.append((roots[keep] ^ m["outputs"][keep]) & 1)
        orig_out.append(a + (roots[(roots >= 0) & (m["outputs"] < 0)] >> 1))
        const_out.append(roots[(roots >= 0) & (m["outputs"] < 0)] & 1 ^ (m["outputs"][(roots >= 0) & (m["outputs"] < 0)] & 1))
    for c in both:
        c.update(prob=np.zeros(len(c["x"]), np.float32), tt_sim=np.zeros(0, np.float32),
                 tt_pair_index=np.zeros((0, 2), np.int64))
    G = deepgate.circuits_to_batch(both, "cuda:0")
    G.tt_pair_index = torch.from_numpy(np.concatenate(pairs).T.copy()).cuda()
    ones, diff, patterns = deepgate.simulate_counts(G, kind, patterns=32768)
    want = np.concatenate(flip) * patterns
    assert np.array_equal(diff.cpu().numpy(), want)
    ones = ones.cpu().numpy()
    # an output that folded to a constant: the original node is constant (const_out: 1 when it reads 1)
    assert np.array_equal(ones[np.concatenate(orig_out).astype(np.int64)], np.concatenate(const_out) * patterns)
    return mapped


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_mapped_copies_simulate_equal_cfg2(kind):
    _check_pairs(synth.make_circuits("aig", 64, (16, 64), (500, 1500), cfg=2), kind)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_mapped_copies_simulate_equal_200k(tmp_path, kind):
    data, A = TA.random_aig(64, 512, 200_000, 800, seed=3)
    c = read_aiger(TA.write(tmp_path, "seq200k.aig", data), "aig")
    m = _check_pairs([c], kind)[0]
    assert sum(gate_arity_counts(m).values()) <= A


@pytest.mark.gpu
def test_batch_independence(tmp_path):
    circuits = _cases(tmp_path)[:16]
    for kind in KINDS:
        together = MP.map_circuits(circuits, kind, "cuda:0", batch_size=16)
        for c, t in zip(circuits, together):
            alone = MP.map_circuits([c], kind, "cuda:0")[0]
            for key in ("x", "edge_index", "outputs", "origin"):
                assert np.array_equal(alone[key], t[key]), key


@pytest.mark.gpu
def test_cli_map_xmg_to_training(tmp_path):
    import types
    import deepgate
    d = tmp_path / "netlists"
    d.mkdir()
    data, A = TA.random_aig(64, 512, 200_000, 800, seed=3)
    TA.write(d, "seq200k.aig", data)
    for i in range(3):
        TA.write(d, "small%d.aig" % i, TA.random_aig(8, 4, 300, 50, seed=4 + i, n_out=8)[0])
    TA.write(d, "adder8.aag", TA.adder(8))
    out = tmp_path / "ds"
    env = dict(os.environ)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env["PYTHONPATH"] = os.pathsep.join([os.path.join(root, "multi-gate-vae_b200"), env.get("PYTHONPATH", "")])
    r = subprocess.run([sys.executable, "-m", "deepgate.simulate", "--aiger", str(d), "--type", "xmg", "--map",
                        "--out", str(out), "--class-pairs", "16"], env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "mapped 5 circuits" in r.stdout and "labelled 5 circuits" in r.stdout, r.stdout
    torch.manual_seed(0)
    parser = deepgate.NpzParser(str(out), str(out / "graphs.npz"), str(out / "labels.npz"), "xmg", random_shuffle=False,
                                trainval_split=0.5)
    train, val = parser.get_dataset()
    codes = torch.cat([g.gate.reshape(-1) for g in list(train) + list(val)]).long()
    for name in ("MAJ", "XOR", "OR"):
        assert int((codes == CODES.index(name)).sum()) > 0, name
    enc = deepgate.digae_layer.DirectMultiGCNEncoder(dim_hidden=64, dim_feature=6, s_rounds=1, t_rounds=1)
    model = deepgate.dg_ae_model_xmg.Model(struct_encoder=enc, dim_hidden=64)
    before = {k: v.detach().clone() for k, v in model.named_parameters()}
    args = types.SimpleNamespace(model="DG_AE", type="xmg")
    trainer = deepgate.Trainer(args, model, training_id="map", save_dir=str(tmp_path / "exp"), device="cuda:0",
                               batch_size=1, distributed=False, rc_prob_func_weight=[1.0, 4.0, 4.0])
    trainer.train(1, train, val)
    log = open(trainer.log_path).read()
    assert "train|" in log and "nan" not in log.lower()
    for sfx in ("maj", "xor", "or"):
        names = [k for k in before if k.startswith("update_%s_func." % sfx)]
        assert names
        after = dict(model.named_parameters())
        assert any(not torch.equal(before[k].cpu(), after[k].detach().cpu()) for k in names), sfx
